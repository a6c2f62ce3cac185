// engine.cuh -- internal interfaces between the stage kernels, the lock-step batch engine and the
// C ABI (capi.cu).  Nothing here is exported.
//
// Every stage kernel takes an ARRAY of device-resident job descriptors and handles job
// blockIdx.{y|z}: the stage entry points of the C ABI run them with one job, the batch engine with
// one job per registration, rewritten on the device by its control kernels between ticks (no host
// round trip inside the RANSAC loops).
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <functional>
#include <vector>

#include "common.cuh"
#include "edge_fmt.cuh"

namespace psulvsb {

// ---- stage 1 --------------------------------------------------------------------------------
struct K1Consts {
  float half_bias;  // c/2, c = beta^2 (1 + 2^-6) (+ rounding head-room): A' = A - c/2, S' = S - c
  float two_beta2;  // 2 beta^2
  float r0;         // 2 beta^2 c - beta^4   ( r = 2 beta^2 S - beta^4 = two_beta2 * S' + r0 )
  float kappa;      // band slope: |v - v_c| <= kappa * S
  float w_thr;      // kappa * c (+slack): pair flagged iff |v| - kappa S' <= w_thr  or  S' <= 0
  double beta;      // FP64 threshold of the exact test
  float beta4;      // beta^4 (fast path: v = D^2 - (2 beta^2 S - beta^4))
  float t_fast;     // fast-path sign is trusted iff |v| > t_fast (rounding band + the a + b <= beta case)
};
K1Consts make_k1_consts(double beta, double coord_bound);

struct K1Job {
  const float4* src;  // packed (centred) points, PAIR-INTERLEAVED (common.cuh il_store): il_records(n) float4 records
  const float4* dst;
  const double* src64;  // column-major 3 x n, original coordinates
  const double* dst64;
  int n, row_begin, row_end;
  K1Consts c;
  uint32_t* mask;
  int stride;                    // words per mask row
  uint32_t* row_counts;          // [n], accumulated with atomicAdd (caller zeroes)
  unsigned long long* border;    // accumulated
  int active;
};

struct CompactJob {
  const uint32_t* mask;
  int n, stride;
  const uint32_t* row_counts;
  unsigned long long* offsets;  // [n+1]
  void* edges;                  // EdgeWide or EdgeNarrow list (edge_fmt.cuh), as the launch says
  unsigned long long cap;
  unsigned long long* n_edges;
  int active;
};

// unknown-scale stage 1 (k1_ratio.cu): ratio histogram and its three-bin reduced set
constexpr double RATIO_MAX_SCALE = 2.0e6;  // largest MaxScale served (a 40 M-bin histogram)
constexpr int RATIO_MAX_GROWTHS = 8;       // each growth more than doubles MaxScale: the 8th passes RATIO_MAX_SCALE
struct RatioJob {
  const double* src64;  // column-major 3 x n
  const double* dst64;
  int n;
  uint32_t* pair_bin;                 // [n (n - 1) / 2] bin of every pair, row-major pair order
  unsigned int* hist;                 // [final MaxScale * 20], zero on entry (sized after phase 0)
  unsigned long long* last;           // same length, zero on entry
  double* row_max;                    // [n - 1] largest ratio of each row (NaN ignored)
  unsigned long long* bp_idx;         // [RATIO_MAX_GROWTHS] growth break points: from pair bp_idx[k] on ...
  double* bp_scale;                   // ... MaxScale == bp_scale[k]
  unsigned int* bp_n;
  double* final_scale;                // MaxScale after the last pair
  unsigned int* peak;                 // [2]: max height, peak bin
  unsigned int* class_counts;         // [3 n]
  unsigned long long* class_offsets;  // [3 n + 1]
  unsigned long long* n_edges;
  void* edges;                        // NULL in phase 0; EdgeWide or EdgeNarrow list, as ratio_emit says
  unsigned long long cap;
  int* bad;                           // written by phase 0: 0, 1 an infinite ratio, 3 final MaxScale > RATIO_MAX_SCALE
  int active;
};

// ---- stage 2 --------------------------------------------------------------------------------
struct SampleJob {
  uint64_t seed;
  uint32_t domain, event;
  unsigned long long n, count, max_draws;
  uint32_t* first;               // [sample_table_words(n, max_draws)] accept bitmask, all zero on entry and on exit
  unsigned long long* chunk_prefix;  // [sample_chunk_slots(max_draws)] accepted draws before each chunk
  unsigned int* ticket;          // zero on entry and on exit (last-CTA-done counter of the bucket pass)
  uint32_t* draws;               // optional cache of the draw values [draws_cap] (16-byte aligned), or NULL
  unsigned long long draws_cap;
  uint32_t* blist;               // optional bucket-list scratch [blist_cap] (k2_sampler.cu), or NULL
  unsigned long long blist_cap;
  unsigned int* bcount;          // [sample_list_counters()] list fill counters + overflow flag, zero on entry and on exit
  uint32_t* out;                 // [count]
  unsigned long long* status;    // draws consumed (0: max_draws too small)
  int identity;                  // 1: out[r] = r (registration.cc:839-847, empty-sample fallback)
  // optional post-processing fused into the emission kernel (batch engine):
  int post;                      // 0 none, 1 endpoint flags of the sampled edges, 2 gather basic edges
  const void* edges;             // post 1/2: the reduced set, EdgeWide or EdgeNarrow (edge_fmt.cuh), as the launch says
  const uint32_t* via;           // post 2: L_sampled (out[r] indexes it)
  uint2* gathered;               // post 2: gathered[r] = edges[via[out[r]]], unpacked (uint2 whatever the list's format)
  const double* pts8;            // post 2, optional: 64-byte point records (sx sy sz tx ty tz 0 0) ...
  double* lv_out;                // ... then the line vector of gathered[r] goes to lv_out[c * lv_cap + r], c = 0..5
  unsigned long long lv_cap;     //     (r < lv_cap): the GNC-TLS kernel finds its line vectors already formed
  uint8_t* flags;                // post 1: [n_points] endpoint flags
  uint32_t* vbits;               // post 1, optional: [ceil(n / 32)] value bitmap, zero on entry and on exit -- the flags
                                 // then come from a streaming pass over the edge list (launch_sample(flag_points > 0))
  int n_points;
  int active;
};

// ---- stage 3 --------------------------------------------------------------------------------
struct GncJob {
  const double* src;     // column-major 3 x n_points
  const double* dst;
  const double* pts8;    // optional [n_points][8]: the same points as 64-byte records (sx sy sz tx ty tz 0 0)
  const uint2* edges;    // K endpoint pairs (a, b): sv = s[b] - s[a], tv = (t[b] - t[a]) * inv_scale
  unsigned long long K;
  double inv_scale;
  double noise_bound;    // already multiplied by 2 / scale (registration.cc:1106-1108)
  double gnc_factor;
  double cost_threshold;
  int max_iterations;
  int use_init;          // 1: first iteration uses R_init (registration.cc:1617-1621)
  double R_init[9];      // column-major
  double* weights;       // K doubles of scratch (overflow beyond the shared-memory capacity)
  double* lv;            // optional SoA scratch [6][lv_cap] for the line vectors beyond that capacity
  unsigned long long lv_cap;
  uint32_t* perm;        // optional [2][lv_cap] index scratch: enables parking sleeping line vectors (k3_rotation.cu)
  int lv_ready;          // 1: lv[c * lv_cap + k], k < min(K, lv_cap), already hold the line vectors (sampler emit pass)
  double* R_out;         // column-major
  uint8_t* inliers;      // [K] or NULL
  uint8_t* point_flags;  // [n_points] or NULL: endpoints of inlier line vectors
  int n_points;
  int* info;             // [4]: iterations, inlier count
  double* cost;
  long long* prof;       // optional [8] diagnostics: pass / loop / SVD cycles, cached count, prologue / epilogue cycles
  // grid mode (more than 8 CTAs per registration): [2][ctas][16] doubles and one counter, see k3_rotation.cu
  double* grid_red;
  unsigned int* grid_bar;
  int active;
};
constexpr int GNC_GRID_RED_DOUBLES = 2 * 16;  // per CTA of a registration in grid mode

// ---- clique escalation (k5_clique.cu) -----------------------------------------------------------
struct CliqueJob {
  const uint2* edges;
  unsigned long long n_edges;
  const double* src;  // filter != 0: keep an edge iff its line vector is length-consistent within beta
  const double* dst;
  double beta;
  int filter;
  int n_vertices;
  uint32_t* adj;  // [clique_scratch_words(n_vertices)] bit matrix scratch + the exact search's work area
  int stride;
  uint8_t* flags;  // [n_vertices] out: clique membership
  int* size;       // out
  int* proven;     // out: 1 = the size is the exact maximum, 0 = the search gave up (greedy answer kept)
  int active;
};
inline size_t clique_scratch_words(int n_vertices) {
  return (((size_t)n_vertices * (size_t)((n_vertices + 31) / 32) + 3) & ~(size_t)3) + 8;
}
// exact = false: the greedy maximal clique only
int launch_max_clique(cudaStream_t st, const CliqueJob* d_jobs, int n_jobs, int max_vertices, int max_stride,
                      unsigned long long max_edges, bool exact);

int launch_knn_normals(cudaStream_t st, const double* pts, int n, int k, const double* viewpoint, double* normals);

// ---- stage launchers (k1_consistency.cu, k2_sampler.cu, k3_rotation.cu, k4_score.cu) -----------
int launch_pack_points(cudaStream_t st, const double* pts, int n, const double center[3], float4* out);
// per-point float4 records -> K1's pair-interleaved records (out: il_records(n) float4)
int launch_interleave_points(cudaStream_t st, const float4* in, int n, float4* out);
// max_n / max_rows: grid extents over all jobs
// row_sectors: EVERY job's mask has stride % 8 == 0 (rows on 32-byte sector boundaries): tiles leave as whole sectors
int launch_consistency_mask(cudaStream_t st, const K1Job* d_jobs, int n_jobs, int max_n, int max_rows, bool row_sectors);
int launch_symmetrize(cudaStream_t st, uint32_t* mask, int n, int stride);
// narrow: the jobs' edge lists are EdgeNarrow (every n <= kEdgeNarrowMaxPoints), else EdgeWide
int launch_compact_edges(cudaStream_t st, const CompactJob* d_jobs, int n_jobs, int max_n, bool scan, bool emit,
                         bool narrow);
// The unknown-scale stage 1 of the jobs rj (device copy d_rj) up to the reduced-set sizes: phase 0, then the final
// MaxScales and refusal flags come back to the host (rj[b].final_scale == rj[0].final_scale + b and rj[b].bad ==
// rj[0].bad + b; `st` is synchronised).  A refused job ends the call with PSULVSB_ERR_UNSUPPORTED.  hist_arena(bytes)
// returns that much device memory (NULL: failed, the message is set) for the histograms, zeroed and laid out here;
// phase 1 runs between the events ev0 and ev1 (either may be NULL) and leaves each size in *rj[b].n_edges.
int ratio_count(cudaStream_t st, std::vector<RatioJob>& rj, RatioJob* d_rj, int max_n,
                const std::function<void*(size_t)>& hist_arena, cudaEvent_t ev0, cudaEvent_t ev1);
// phase 2: every job's reduced set (rj[b].edges, rj[b].cap) in reference order, EdgeNarrow lists if `narrow`
int ratio_emit(cudaStream_t st, const std::vector<RatioJob>& rj, RatioJob* d_rj, int max_n, bool narrow);

// Draw budget for `count` distinct values out of n by rejection (mean + 8 sigma; coupon collector
// tail for count == n).  Same formula on host and device so both agree on the stream window.
__host__ __device__ inline unsigned long long sample_max_draws_formula(unsigned long long n,
                                                                       unsigned long long count) {
  if (n == 0 || count == 0) return 0;
  if (count > n) count = n;
  double e;
  if (count == n) {
    e = (double)n * (log((double)n) + 0.5772156649 + 10.0);
  } else {
    const double f = (double)count / (double)n;
    const double mean = -(double)n * log1p(-f);
    e = mean * 1.02 + 8.0 * sqrt(mean + 1.0) + 64.0;
  }
  unsigned long long m = (unsigned long long)e + 8;
  m = (m + 3) & ~3ull;
  if (m > 0xFFFFFFF0ull) m = 0xFFFFFFF0ull;
  return m;
}
unsigned long long sample_default_max_draws(unsigned long long n, unsigned long long count);
unsigned long long sample_chunk_slots(unsigned long long max_draws);
unsigned long long sample_list_entries(unsigned long long n, unsigned long long max_draws);  // 0: lists not applicable
unsigned long long sample_list_counters();
unsigned long long sample_table_words(unsigned long long n, unsigned long long max_draws);
// true: launch_sample with this n_bound draws its jobs on chip (all but the (1.0, 1.0) escalation's long windows),
// without the draw cache and bucket lists
bool sample_onchip_bound(unsigned long long n_bound);
// flag_points > 0: the post-1 jobs' endpoint flags come from the flag pass (SampleJob::vbits), n_points <= flag_points;
// narrow: the jobs' SampleJob::edges are EdgeNarrow lists, else EdgeWide
int launch_sample(cudaStream_t st, const SampleJob* d_jobs, int n_jobs, unsigned long long max_draws_bound,
                  unsigned long long n_bound, int flag_points = 0, bool narrow = false);
int launch_philox_fill(cudaStream_t st, uint64_t seed, uint32_t domain, uint32_t event, unsigned long long first_k,
                       unsigned long long count, uint32_t* out);

int gnc_default_capacity();
int gnc_cluster_for(int n_jobs);
// max_points > 0 allows the point-cache mode of the single-CTA variant (upper bound of GncJob::n_points)
int launch_gnc_tls(cudaStream_t st, const GncJob* d_jobs, int n_jobs, int cap_per_cta, int cluster, int n_active = 0);
int launch_kabsch_batch(cudaStream_t st, const double* src, const double* dst, const uint2* edges,
                        const uint32_t* sets, int k, unsigned long long n_hyp, double* R, double* t);

int launch_tls_translation(cudaStream_t st, const double* src, const double* dst, const uint8_t* flags, int n,
                           double scale, const double* R, double noise, const double* last_best, double* t_out,
                           int* n_points);
int launch_score_one(cudaStream_t st, const double* src, const double* dst, int n, double scale, const double* R,
                     const double* t, double tau, uint8_t* inliers, double* residuals, int* count);
int launch_score_batch(cudaStream_t st, const float4* src, const float4* dst, const double* src64, const double* dst64,
                       int n, const double* hyp, unsigned long long n_hyp, unsigned long long hyp_begin, double scale,
                       double tau, double coord_bound, const double* csrc, const double* cdst, uint32_t* counts,
                       unsigned long long* best, unsigned long long* border);

// ---- multi-GPU plumbing (comm.cu) -------------------------------------------------------------------
struct Comm;
int comm_unique_id(void* out128);
int comm_create(Comm** out, int device, int rank, int world, const void* id128);
void comm_destroy(Comm* c);
int comm_rank(const Comm* c);
int comm_world(const Comm* c);
int comm_allreduce_sum_u32(Comm* c, cudaStream_t st, uint32_t* d_inout, size_t n);
int comm_allreduce_max_u64(Comm* c, cudaStream_t st, unsigned long long* d_inout, size_t n);
int comm_allgather_u64(Comm* c, cudaStream_t st, const unsigned long long* d_send, unsigned long long* d_recv);
int comm_allgatherv_inplace_u32(Comm* c, cudaStream_t st, uint32_t* base, const unsigned long long* offsets);
void triangular_row_range(int n, int rank, int world, int* begin, int* end);

// ---- batch engine pool (engine.cu) --------------------------------------------------------------
class EnginePool;
int pool_create(EnginePool** out, int device);
void pool_destroy(EnginePool* p);
int pool_set_batching(EnginePool* p, int chunk, int lanes);
int pool_set_host_threads(EnginePool* p, int n);
int pool_solve_one(EnginePool* p, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                   psulvsb_solution_t* solution, psulvsb_trace_t* trace);
int pool_solve_batch(EnginePool* p, const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B,
                     const uint64_t* seeds, psulvsb_solution_t* solutions);
int pool_submit(EnginePool* p, const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B,
                const uint64_t* seeds, psulvsb_solution_t* solutions, uint64_t* ticket);
int pool_wait(EnginePool* p, uint64_t ticket);
int pool_upload(EnginePool* p, const psulvsb_problem_t* problems, int B);
// ONE registration whose consistency rows are sharded over the ranks of `comm` (every rank passes the same problem and
// gets the same solution)
int pool_solve_sharded(EnginePool* p, Comm* comm, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                       psulvsb_solution_t* solution, psulvsb_trace_t* trace);
int pool_solve_resident(EnginePool* p, const psulvsb_params_t* params, const uint64_t* seeds,
                        psulvsb_solution_t* solutions, psulvsb_trace_t* trace_first);
int pool_batch_size(const EnginePool* p);
int pool_last_ticks(const EnginePool* p);
int pool_last_chunk_ticks(const EnginePool* p, int* out, int cap);
long long pool_launch_count(const EnginePool* p);
double pool_last_device_ms(const EnginePool* p);
double pool_last_stage_ms(const EnginePool* p, int which);

}  // namespace psulvsb
