/*
 * psulvsb.h -- C ABI of the B200-native PSULVSB registration hot path (libpsulvsb_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, int status codes, no C++/torch types.
 * It replaces, for the PSULVSB path only, what a binding to the reference would call:
 *
 *   teaser::RobustRegistrationSolver::Params                     (registration.h:378-473)
 *   teaser::RobustRegistrationSolver::RobustRegistrationSolver   (registration.cc:465-468)
 *   teaser::RobustRegistrationSolver::solve(src, dst)            (registration.cc:622-1535)
 *   teaser::RobustRegistrationSolver::getSolution()              (registration.h:553)
 *   teaser::RegistrationSolution                                 (registration.h:34-41)
 *
 * plus stage-level entry points for the four CUDA stages (device pointers + stream), which the
 * parity tests and the benchmark drive directly.  Matrices follow Eigen's default layout:
 * a 3xN point set is a column-major double[3*N] (== Eigen::Matrix<double,3,Dynamic>::data()).
 *
 * All functions return PSULVSB_OK (0) or an error code; psulvsb_last_error() gives the message
 * of the last failure on the calling thread.  Nothing throws across this boundary.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with
 * PSULVSB_ERR_NO_DEVICE.
 */
#ifndef PSULVSB_H_
#define PSULVSB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSULVSB_VERSION 100 /* 0.1.0 */

enum {
  PSULVSB_OK = 0,
  PSULVSB_ERR_INVALID = 1,     /* bad argument                                                  */
  PSULVSB_ERR_CUDA = 2,        /* CUDA runtime failure (see psulvsb_last_error)                 */
  PSULVSB_ERR_NO_DEVICE = 3,   /* no usable sm_100 device                                       */
  PSULVSB_ERR_CAPACITY = 4,    /* a caller-provided buffer is too small                         */
  PSULVSB_ERR_UNSUPPORTED = 5, /* configuration outside the implemented hot path                */
  PSULVSB_ERR_INTERNAL = 6
};

/* Philox sample-stream domains (DESIGN.md "Sample stream").  A draw is addressed by
 * (seed, domain, event, k); nothing depends on how many draws other events consumed. */
enum {
  PSULVSB_DOMAIN_L_SAMPLED = 1, /* registration.cc:852-861, event = host round                  */
  PSULVSB_DOMAIN_BASIC = 2,     /* registration.cc:916-932, event = global local-iteration index */
  PSULVSB_DOMAIN_UNIFORM = 3,   /* registration.cc:604-609 draws at :1428/:1438, k = point index */
  PSULVSB_DOMAIN_SCALE = 4,     /* registration.cc:90                                           */
  PSULVSB_DOMAIN_TUPLE = 5      /* matcher tuple test, event 0, k = 3 trial + corner (psulvsb_match_host) */
};

/* ---- Params: RobustRegistrationSolver::Params (registration.h:378-473) plus the reference's
 * compile-time constants and in-loop overrides lifted into fields (defaults = reference values,
 * see psulvsb_default_params). ori_src / ori_dst / keep_mask / reduce_map travel in
 * psulvsb_problem_t because they are per-problem data. */
typedef struct psulvsb_params {
  double noise_bound;             /* registration.h:383                                         */
  double cbar2;                   /* registration.h:388                                         */
  int estimate_scaling;           /* registration.h:396; 1 = ratio histogram + TLS scale (:687-752, :958-983) */
  int rotation_max_iterations;    /* registration.h:416                                         */
  double rotation_gnc_factor;     /* registration.h:411                                         */
  double rotation_cost_threshold; /* registration.h:426                                         */
  int inlier_selection_mode;      /* registration.h:365-370 (0 PMC_EXACT .. 3 NONE)             */
  double kcore_heuristic_threshold;
  double score_noise_bound;       /* registration.cc:33  NOISE_BOUND; PrNoise = 2x (:36)        */
  double inloop_noise_bound;      /* registration.cc:938                                        */
  double inloop_cbar2;            /* registration.cc:939                                        */
  int inloop_max_iterations;      /* registration.cc:941                                        */
  double inloop_gnc_factor;       /* registration.cc:942                                        */
  double inloop_cost_threshold;   /* registration.cc:945                                        */
  double rotation_similar;        /* registration.cc:48                                         */
  int local_max_iter;             /* registration.cc:49                                         */
  double tpro_host;               /* registration.cc:772                                        */
  double tpro_local;              /* registration.cc:898                                        */
  int host_round_limit;           /* registration.cc:781                                        */
  double wallclock_cap_s;         /* registration.cc:1475; <= 0 disables (replay mode)          */
  int self_update;                /* registration.cc:786-832 on/off                             */
  uint64_t seed;                  /* Philox key of the sample stream                            */
} psulvsb_params_t;

/* One registration problem, host pointers (reference: the arguments of solve() plus the four
 * PSULVSB Params fields, registration.h:469-472). */
typedef struct psulvsb_problem {
  const double* src;     /* 3xC column-major: reduced source correspondences                    */
  const double* dst;     /* 3xC                                                                 */
  int C;
  const double* ori_src; /* 3xM: Params::ori_src                                                */
  const double* ori_dst; /* 3xM: Params::ori_dst                                                */
  int M;
  const int* keep_mask;  /* [M] in {-1,0,1}: Params::keep_mask                                  */
  const int* reduce_map; /* [M] reduced column of original j, -1 if absent (dense form of the   */
                         /*     reference's std::map<int,int> Params::reduce_map)               */
} psulvsb_problem_t;

/* RegistrationSolution (registration.h:34-41) + diagnostics. */
typedef struct psulvsb_solution {
  int valid;
  double scale;
  int final_inlier_count;
  double translation[3];
  double rotation[9]; /* column-major, == Eigen::Matrix3d::data()                               */
  int host_rounds;
  int local_iters;
  long long n_line_vectors; /* C(C-1)/2                                                         */
  long long n_reduced;      /* |L_reduced| after the one-time consistency pass                  */
  int final_C;              /* working-set size after self-update appends                       */
  int refined;              /* weighted-SVD refinement accepted (registration.cc:1516)          */
  int escalations;          /* rate escalations taken (registration.cc:1377-1388)               */
  long long borderline_pairs; /* K1 pairs re-evaluated in FP64 (inside the FP32 error band)     */
  int status;               /* PSULVSB_OK or the per-problem error                              */
} psulvsb_solution_t;

/* Per local-iteration / per host-scoring trace records (same content as the oracle's, so parity
 * tests can compare the two solvers step by step). */
typedef struct psulvsb_local_trace {
  int host_round, local_iter, n_sampled_lines, n_sampled_points, basic_choose, gnc_iterations;
  int rot_inliers, n_rot_points, similar, curr_count, best_count, local_r;
  double p_local, l_rate, b_rate, scale;
  double R[9];
  double t[3];
} psulvsb_local_trace_t;

typedef struct psulvsb_host_trace {
  int host_round, curr_count, best_host, new_corr_count, inlier_map_size, host_r;
  double p_host;
} psulvsb_host_trace_t;

typedef struct psulvsb_trace {
  psulvsb_local_trace_t* local;
  int local_cap, local_n;
  psulvsb_host_trace_t* host;
  int host_cap, host_n;
  int* final_inliers;  /* optional [M]                                                          */
  int* inlier_counter; /* optional [M]                                                          */
  int* reduce_map_out; /* optional [M]: reduce_map after self-update (column of each original
                          correspondence in the grown working set, -1 = absent): entries >= C are the
                          columns the reference appends to the caller's src / dst (registration.cc:800-806) */
} psulvsb_trace_t;

typedef struct psulvsb_handle_s* psulvsb_handle_t;

/* ------------------------------------------------------------------------------------------ */
/* lifecycle                                                                                   */
/* ------------------------------------------------------------------------------------------ */
int psulvsb_version(void);
const char* psulvsb_last_error(void);
void psulvsb_default_params(psulvsb_params_t* p);
/* Number of CUDA devices the library can use (0 when none; never fails). */
int psulvsb_device_count(void);
/* One handle = one device and a small pool of lock-step engines (each its own stream and private device arenas);
 * handles are independent and may be used from different threads (the reference's solver is neither re-entrant nor
 * thread safe, registration.cc:40-50). */
int psulvsb_create(psulvsb_handle_t* out, int device);
/* How a batch is advanced.  chunk: registrations per lock-step chunk (0 = one per SM of the device); lanes: chunks in
 * flight at once, each on its own engine, stream and host thread (0 = 4).  A batch of at most `chunk` problems runs as
 * one chunk.  With host buffers (psulvsb_solve_batch) chunks are handed to the lanes dynamically, so chunk k + 1 is
 * staged and copied while chunk k is solved; a resident batch is split evenly over at most `lanes` engines.  Results
 * never depend on these settings (every registration has its own state and sample stream).  Changing them drops the
 * resident batch. */
int psulvsb_set_batching(psulvsb_handle_t h, int chunk, int lanes);
/* Host threads the handle may use for staging uploads (psulvsb_solve_batch / psulvsb_batch_upload copy the caller's
 * arrays into pinned memory while earlier groups are already on their way to the device).  0 = the CPUs available to
 * the process (its affinity mask).  On a multi-GPU node give every rank its share (cores / ranks). */
int psulvsb_set_host_threads(psulvsb_handle_t h, int n);
/* Debug / test switches (process-wide; the library reads NO environment variable).  They select among code paths
 * that produce identical results: "gnc_deep_margin" (rad), "gnc_prefetch", "gnc_cluster" (1 / 2 / 4 / 8 CTAs per
 * registration), "gnc_cps", "gnc_park_pct", "gnc_grid_lv" (line vectors per CTA above which GNC-TLS spreads one
 * registration over the grid), "sample_list_cap_test", "k1_variant" (1..4 rows per thread), "upload_prof" (1: phase
 * timings on stderr), "edge_wide" (1: 8-byte reduced-set edges even where 4-byte ones fit), "reset" (all back to
 * defaults). */
int psulvsb_debug_set(const char* name, double value);
int psulvsb_destroy(psulvsb_handle_t h);

/* ------------------------------------------------------------------------------------------ */
/* end-to-end: RobustRegistrationSolver(params).solve(src, dst); getSolution()                 */
/* ------------------------------------------------------------------------------------------ */
/* Host buffers in, host solution out (H2D, all stages, D2H inside the call). */
int psulvsb_solve(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                  psulvsb_solution_t* solution, psulvsb_trace_t* trace /* may be NULL */);
/* B independent problems advanced in lock step on the device (batched registration mode).
 * seeds: optional per-problem Philox keys (default params->seed + index). */
int psulvsb_solve_batch(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problems,
                        int B, const uint64_t* seeds, psulvsb_solution_t* solutions);
/* A STREAM of batches, pipelined.  psulvsb_batch_submit queues the batch and returns at once with a ticket;
 * psulvsb_batch_wait(ticket) returns when its solutions are written (tickets may be waited for in any order, each
 * once).  Everything the call was given -- the problem records, the point arrays they reference, seeds, solutions --
 * must stay valid and untouched until the wait has returned; params is copied.  The handle's lanes pull lock-step
 * chunks from ONE queue across calls; at most `lanes` chunks are being solved at a time and one more worker stages and
 * copies the next chunk meanwhile, so with lanes + 1 batches (or chunks) in flight the uploads run under the solves and
 * cost nothing (psulvsb_solve_batch, which must drain the device before it returns, pays for them).  Results are those of psulvsb_solve_batch.  Every other call on the handle first waits
 * for the queue to empty.  (The reference solves one pair at a time on one thread: PSULVSB.cc:326-331.) */
int psulvsb_batch_submit(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problems,
                         int B, const uint64_t* seeds, psulvsb_solution_t* solutions, uint64_t* ticket);
int psulvsb_batch_wait(psulvsb_handle_t h, uint64_t ticket);
/* Resident variant: upload once, then solve the resident batch any number of times (inputs stay
 * in HBM; only the solutions come back).  Used for the device-resident throughput figure. */
int psulvsb_batch_upload(psulvsb_handle_t h, const psulvsb_problem_t* problems, int B);
/* n_solutions: capacity of `solutions`; must equal the resident batch size (psulvsb_batch_resident_size), which
 * every upload / psulvsb_solve / psulvsb_solve_batch on the handle replaces -- a mismatch is PSULVSB_ERR_INVALID. */
int psulvsb_batch_solve_resident(psulvsb_handle_t h, const psulvsb_params_t* params, const uint64_t* seeds,
                                 psulvsb_solution_t* solutions, int n_solutions);
/* Problems currently resident on the handle (0: nothing uploaded, or the last upload failed). */
int psulvsb_batch_resident_size(psulvsb_handle_t h);
/* Kernel launches issued by the handle since creation / device time (ms) of the last solve call: CUDA events,
 * from the start of the call to the end of its last chunk (the chunks run on the engines' own streams). */
long long psulvsb_launch_count(psulvsb_handle_t h);
double psulvsb_last_device_ms(psulvsb_handle_t h);
/* Device time (ms), CUDA events on the engines' streams, of part `which` of the last solve call:
 * 0 stage 1 in full (float4 packing, mask, row scan, n_red read-back, edge compaction, state init), mean over chunks,
 * 1 the tick loop (sampling, GNC-TLS, translation, scoring, control), mean over chunks,
 * 2 the consistency-mask kernel alone: time during which the launch of SOME chunk was running (union of the
 *   launches' intervals; one launch per chunk),
 * 3 the GNC-TLS launches of all ticks, union over chunks likewise, 4 refinement + solution copy, mean over chunks. */
double psulvsb_last_stage_ms(psulvsb_handle_t h, int which);
/* Engine ticks (lock-step local iterations of a chunk) of the last solve call: the largest over its chunks ... */
int psulvsb_last_ticks(psulvsb_handle_t h);
/* ... and per chunk: writes min(cap, n_chunks) entries, returns n_chunks. */
int psulvsb_last_chunk_ticks(psulvsb_handle_t h, int* out, int cap);

/* ------------------------------------------------------------------------------------------ */
/* stage entry points: DEVICE pointers, asynchronous on `stream` (a cudaStream_t, may be NULL) */
/* ------------------------------------------------------------------------------------------ */

/* Points: column-major double 3xN -> float4 (x-cx, y-cy, z-cz, 0).  center may be NULL (0). */
int psulvsb_pack_points(void* stream, const double* d_pts, int n, const double center[3], void* d_out_float4);

/* Stage 1 -- line-vector length-consistency mask (registration.cc:693-732 + :418-434).
 * bit j of row i (word j>>5 of d_mask + i*row_stride_words) is set iff j > i and
 * | |s_j-s_i| - |t_j-t_i| | <= beta evaluated exactly as the FP64 reference does: the kernel
 * evaluates in FP32 from the float4 tiles and re-evaluates every pair inside the rigorous FP32
 * error band in FP64 from d_src64/d_dst64, counting them in *d_border_count.
 * coord_bound: max |coordinate| over the float4 inputs (sets the band).
 * d_row_counts[n] receives the popcount of each (upper-triangular) row. */
int psulvsb_consistency_mask(void* stream, const void* d_src_f4, const void* d_dst_f4, const double* d_src64,
                             const double* d_dst64, int n, double beta, double coord_bound, uint32_t* d_mask,
                             int row_stride_words, uint32_t* d_row_counts, unsigned long long* d_border_count);
/* Rows [row_begin, row_end) only (row-block sharding across GPUs; same layout, same bits). */
int psulvsb_consistency_mask_rows(void* stream, const void* d_src_f4, const void* d_dst_f4, const double* d_src64,
                                  const double* d_dst64, int n, int row_begin, int row_end, double beta,
                                  double coord_bound, uint32_t* d_mask, int row_stride_words,
                                  uint32_t* d_row_counts, unsigned long long* d_border_count);
/* Mirror the upper triangle into the lower one (full symmetric adjacency, zero diagonal). */
int psulvsb_mask_symmetrize(void* stream, uint32_t* d_mask, int n, int row_stride_words);
/* Reduced set in reference order (registration.cc:756-766): edges[k] = (i, j), i < j, row-major.
 * d_row_offsets[n+1] (u64) receives the exclusive scan of d_row_counts; *d_n_edges the total. */
int psulvsb_compact_edges(void* stream, const uint32_t* d_mask, int n, int row_stride_words,
                          const uint32_t* d_row_counts, unsigned long long* d_row_offsets, void* d_edges_uint2,
                          unsigned long long edge_capacity, unsigned long long* d_n_edges);
/* Unknown-scale stage 1 (estimate_scaling = true, registration.cc:687-752): the length-ratio histogram with the
 * reference's mid-loop growth of MaxScale, its peak ("the first bin to reach the maximum height") and the reduced set
 * (bins peak, peak - 1, peak + 1, each in pair order) -- the solve's own code.  Synchronous on `stream`.
 * d_pair_bin (optional): n (n - 1) / 2 bins, row-major pair order (i < j).  d_edges_uint2 (optional, NULL = count
 * only): the reduced set as (i, j) pairs; fewer than *n_edges slots is PSULVSB_ERR_CAPACITY with *n_edges set.
 * Host outputs: *n_edges, *max_scale (the final MaxScale, may be NULL), peak[2] = {max height, peak bin} (may be
 * NULL).  NULL arrays / n_edges or n < 2: PSULVSB_ERR_INVALID before any device work; an infinite ratio or a final
 * MaxScale above 2e6: PSULVSB_ERR_UNSUPPORTED, as in psulvsb_solve. */
int psulvsb_ratio_reduced_set(void* stream, const double* d_src64, const double* d_dst64, int n, uint32_t* d_pair_bin,
                              void* d_edges_uint2, unsigned long long edge_capacity, unsigned long long* n_edges,
                              double* max_scale, unsigned int peak[2]);

/* Stage 2 -- replayable sampling without replacement (registration.cc:852-861, :916-932):
 * d_out[r] = r-th distinct value of rand31(seed, domain, event, k) % n, k = 0,1,2,...
 * max_draws = 0 selects psulvsb_sample_default_max_draws(n, count) (mean + 8 sigma of the rejection loop).
 * d_work: >= psulvsb_sample_workspace_bytes(n, count, max_draws) bytes of scratch (16-byte aligned).
 * d_status[0] = draws consumed, i.e. the stream position the sequential loop would be at
 * (0 if max_draws was too small: call again with a larger max_draws).  n < 2^31, max_draws < 2^32. */
unsigned long long psulvsb_sample_workspace_bytes(unsigned long long n, unsigned long long count,
                                                  unsigned long long max_draws);
unsigned long long psulvsb_sample_default_max_draws(unsigned long long n, unsigned long long count);
int psulvsb_sample(void* stream, uint64_t seed, uint32_t domain, uint32_t event, unsigned long long n,
                   unsigned long long count, unsigned long long max_draws, uint32_t* d_out, void* d_work,
                   unsigned long long* d_status);
/* Raw stream access for replay checks. */
int psulvsb_philox_fill(void* stream, uint64_t seed, uint32_t domain, uint32_t event, unsigned long long first_k,
                        unsigned long long count, uint32_t* d_out_rand31);

/* Stage 3a -- GNC-TLS rotation over K line vectors given as endpoint pairs into a point set
 * (registration.cc:1563-1692 + utils.h:121-136).  d_edges: uint2[K] (a, b): sv = s[b]-s[a].
 * R_init: device pointer to a column-major warm start or NULL (first_time).
 * Outputs: d_R[9] column-major, d_inliers[K] (u8), d_info[4] = {iterations, inlier count, 0, 0},
 * d_cost[1].  d_weights: K doubles of scratch. */
int psulvsb_gnc_tls_rotation(void* stream, const double* d_src64, const double* d_dst64, const void* d_edges_uint2,
                             unsigned long long K, double inv_scale, double noise_bound, int max_iterations,
                             double gnc_factor, double cost_threshold, const double* d_R_init, double* d_weights,
                             double* d_R, uint8_t* d_inliers, int* d_info, double* d_cost);
/* Stage 3a, batched: n_jobs independent GNC-TLS solves over one point set, job b using the K endpoint pairs
 * d_edges[b*K .. b*K+K) -- the shape of one engine tick (one basic subset per registration), and the entry the
 * GNC micro-benchmark (profiles/tools/gnc_batch.py) drives.  cluster: CTAs per job (1, 2, 4, 8; 0 = the engine's
 * choice for n_jobs).  d_weights: n_jobs*K doubles of scratch; d_lv: optional n_jobs*6*lv_cap doubles of scratch
 * for the line vectors beyond the shared-memory capacity (NULL: they are re-formed from the points); d_perm:
 * optional n_jobs*2*lv_cap uint32 of scratch (with d_lv: lets the kernel park sleeping line vectors).
 * Outputs: d_R[n_jobs*9] column-major, d_inliers[n_jobs*K] (u8, optional), d_info[n_jobs*4] (iterations, inliers, SVD cycles/16, loop cycles/16),
 * d_prof[n_jobs*8] optional diagnostics (cycles of thread 0: line-vector passes, iteration loop, SVDs; cached line
 * vectors per CTA; prologue and epilogue cycles). */
int psulvsb_gnc_tls_rotation_batch(void* stream, const double* d_src64, const double* d_dst64, int n_points,
                                   const void* d_edges_uint2, unsigned long long K, int n_jobs, double noise_bound,
                                   int max_iterations, double gnc_factor, double cost_threshold, int cluster,
                                   double* d_weights, double* d_lv, unsigned long long lv_cap, uint32_t* d_perm,
                                   double* d_R, uint8_t* d_inliers, int* d_info, long long* d_prof);
/* Stage 3b -- batched closed-form Kabsch, one warp per hypothesis (utils.h:121-136): hypothesis h
 * uses the k line vectors d_sets[h*k .. h*k+k) (indices into d_edges).  Outputs d_R[h*9..]
 * (column-major) and, if d_t != NULL, the translation of the centroid of the sampled endpoints. */
int psulvsb_kabsch_batch(void* stream, const double* d_src64, const double* d_dst64, const void* d_edges_uint2,
                         const uint32_t* d_sets, int k, unsigned long long n_hyp, double* d_R, double* d_t);

/* Max-stabbing translation (registration.cc:436-463 + :121-203) over the points flagged in
 * d_point_flags[n]; d_last_best = NULL when first_time.  d_t_out[3]. */
int psulvsb_tls_translation(void* stream, const double* d_src64, const double* d_dst64, const uint8_t* d_point_flags,
                            int n, double scale, const double* d_R, double noise, const double* d_last_best,
                            double* d_t_out, int* d_n_points);

/* ---- The reference's public sub-solver calls on HOST buffers --------------------------------------------
 * (teaser/include/teaser/registration.h:107-317; what rotation-solver-test.cc, scale-solver-test.cc,
 * translation-solver-test.cc, tls-test.cc and RobustRegistrationSolver::solveForScale / solveForRotation /
 * solveForTranslation / computeTIMs call).  Column-major 3 x n doubles in, results out; each call stages its
 * arrays on the device and runs the kernels the engine runs.  include/teaser/registration.h wraps them in the
 * reference's class names. */

/* RobustRegistrationSolver::computeTIMs (registration.cc:471-505): tims[3 x n(n-1)/2], column
 * i*n - i(i+1)/2 + (j-i-1) = v_j - v_i; map (2 x L ints: i, j) may be NULL. */
int psulvsb_compute_tims_host(const double* pts, int n, double* tims, int* map);
/* ScaleInliersSelector::solveForScale (registration.cc:418-434): inliers[l] = | |src_l| - |dst_l| | <= 2 noise_bound
 * sqrt(cbar2); the scale it reports is 1. */
int psulvsb_scale_inliers_host(const double* src_tims, const double* dst_tims, unsigned long long n, double noise_bound,
                               double cbar2, unsigned char* inliers);
/* TLSScaleSolver::solveForScale (registration.cc:397-415 -> ScalarTLSEstimator::estimate :66-120).  The reference
 * draws candidates with rand(); here draw k of the call is philox(seed; PSULVSB_DOMAIN_SCALE, event, k).
 * last_best_scale: NULL on the first call (first_time), else the reference's scale_last_best. */
int psulvsb_tls_scale_host(const double* src_tims, const double* dst_tims, int n, double noise_bound, double cbar2,
                           uint64_t seed, uint32_t event, const double* last_best_scale, double* scale,
                           unsigned char* inliers);
/* GNCTLSRotationSolver::solveForRotation (registration.cc:1563-1692 + utils.h:121-136).  R_last_best: NULL on the
 * first call, else the warm start (column-major).  R[9] column-major; inliers / cost / iterations may be NULL. */
int psulvsb_gnc_tls_rotation_host(const double* src_tims, const double* dst_tims, unsigned long long n,
                                  double noise_bound, int max_iterations, double gnc_factor, double cost_threshold,
                                  const double* R_last_best, double* R, unsigned char* inliers, double* cost,
                                  int* iterations);
/* TLSTranslationSolver::solveForTranslation (registration.cc:436-463 -> :121-203): per-axis max-stabbing of
 * (dst - src) +- noise_bound sqrt(cbar2); inliers = within the bound of the estimate on all three axes.
 * t_last_best: NULL on the first call, else the pseudo-measurement of :136-161. */
int psulvsb_tls_translation_host(const double* src, const double* dst, int n, double noise_bound, double cbar2,
                                 const double* t_last_best, double* t, unsigned char* inliers);

/* Surface normals by k-nearest-neighbour PCA, what the reference driver gets from PCL before its timed region
 * (examples/teaser_cpp_ply/PSULVSB.cc:35-85: NormalEstimation, setKSearch(20), viewpoint (0,0,0)) and feeds to
 * the histogram pre-filter (psulvsb_io.h).  d_pts / d_normals: column-major 3xn doubles on the device;
 * 3 <= k <= 32; viewpoint may be NULL (origin).  The _host variant takes host buffers (copies inside). */
int psulvsb_estimate_normals(void* stream, const double* d_pts, int n, int k, const double viewpoint[3],
                             double* d_normals);
int psulvsb_estimate_normals_host(const double* pts, int n, int k, const double viewpoint[3], double* normals);

/* ---- Correspondences from two raw clouds (DESIGN.md section 10): what upstream TEASER++ gets from
 * teaser::FPFHEstimation (PCL radius normals + FPFHEstimation) and teaser::Matcher (FLANN + FGR's AdvancedMatching).
 * Parity with PCL / FLANN is unpinned; the tests compare with a numpy restatement (oracle/features.py).
 *
 * FPFH descriptors: points are column-major 3xn doubles; normals from the FP64 covariance of the normal_radius
 * neighbourhood (the point included; fewer than 3 points: NaN), flipped towards the viewpoint (NULL: origin); the
 * 33-bin descriptor of every point over its feature_radius neighbourhood, n x 33 floats row-major (the layout of
 * std::vector<pcl::FPFHSignature33>).  An isolated point gets an all-zero descriptor.  Results are bit-identical from
 * call to call.  d_work: psulvsb_fpfh_workspace_bytes(n) bytes of device scratch (depends on n only); d_normals may
 * be NULL.  Radii must be finite and > 0 (PSULVSB_ERR_INVALID otherwise, before any device work). */
unsigned long long psulvsb_fpfh_workspace_bytes(int n);
int psulvsb_fpfh(void* stream, const double* d_pts, int n, double normal_radius, double feature_radius,
                 const double viewpoint[3], void* d_work, double* d_normals, float* d_features);
int psulvsb_fpfh_host(const double* pts, int n, double normal_radius, double feature_radius,
                      const double viewpoint[3], double* normals, float* features);
/* Two-way nearest neighbour in descriptor space (exact squared L2 over the 33 floats, ties to the lowest index):
 * d_nn_src_to_tgt[i] = nearest target of source descriptor i, d_nn_tgt_to_src[j] = nearest source of target j
 * (-1 when the other side is empty). */
int psulvsb_feature_nn(void* stream, const float* d_fs, int n_src, const float* d_ft, int n_tgt,
                       int* d_nn_src_to_tgt, int* d_nn_tgt_to_src);
/* Matcher::calculateCorrespondences on host buffers: descriptors -> two-way NN -> the list (crosscheck: mutual pairs
 * in ascending source index; otherwise (i, nn(i)) for every i that is some target's nearest source, then (nn(j), j)
 * for every target j) -> optionally the tuple test (up to 1000 triangles whose three edge-length ratios lie in
 * (tuple_scale, 1/tuple_scale), trials drawn from philox(seed; PSULVSB_DOMAIN_TUPLE)).  pairs: room for `capacity`
 * (source, target) index pairs, interleaved; *n_pairs receives the count (also when it exceeds the capacity:
 * PSULVSB_ERR_CAPACITY). */
int psulvsb_match_host(const double* src_pts, int n_src, const double* tgt_pts, int n_tgt, const float* fs,
                       const float* ft, int crosscheck, int tuple_test, double tuple_scale, uint64_t seed, int* pairs,
                       long long capacity, long long* n_pairs);

/* ---- Correspondences for a batch in one call (DESIGN.md section 10, "Batches").  The clouds / pairs array is a HOST
 * array, read before the call returns; its data pointers are device pointers for the asynchronous variants and host
 * pointers for _host.  The radii and the matcher's flags are shared; the viewpoint and the seed belong to each item.
 * Every launch covers the whole batch.  Item b's output is bit-identical to what psulvsb_fpfh_host (with its
 * viewpoint) or psulvsb_match_host (with its seed) returns for it alone, whatever else is in the batch and in which
 * order.  PSULVSB_ERR_INVALID before any device work for B < 0, radii that are not finite and > 0, a negative size, a
 * NULL pointer of an item that is not empty, a non-finite tuple_scale with the tuple test, or a required NULL output;
 * PSULVSB_ERR_UNSUPPORTED when the sizes (n; n_src or n_tgt) add up to 2^31 or more.  B = 0 does nothing. */
typedef struct psulvsb_fpfh_cloud {
  const double* pts;  /* 3 x n, column-major                                                              */
  int n;
  double viewpoint[3]; /* normals flip towards it; zeros = the origin, as NULL does for psulvsb_fpfh        */
} psulvsb_fpfh_cloud_t;
/* Device scratch of psulvsb_fpfh_batch (depends on the sizes only); 0 for B <= 0 or a negative size. */
unsigned long long psulvsb_fpfh_batch_workspace_bytes(const psulvsb_fpfh_cloud_t* clouds, int B);
/* Cloud c's descriptors are rows [sum_{a<c} n_a, ...) of the (sum n) x 33 floats d_features, its normals the same rows
 * of the (sum n) x 3 doubles d_normals (may be NULL).  Asynchronous on `stream`. */
int psulvsb_fpfh_batch(void* stream, const psulvsb_fpfh_cloud_t* clouds, int B, double normal_radius,
                       double feature_radius, void* d_work, double* d_normals, float* d_features);
/* The same on host buffers, synchronous (normals may be NULL). */
int psulvsb_fpfh_batch_host(const psulvsb_fpfh_cloud_t* clouds, int B, double normal_radius, double feature_radius,
                            double* normals, float* features);

/* ---- Surface normals alone (DESIGN.md section 10, "Normals alone"), on FPFH's grid: O(n * neighbourhood) instead of
 * the O(n^2) psulvsb_estimate_normals.  Points and normals are column-major 3xn doubles.
 *   max_nn = 0:      radius neighbourhood, every point within `radius` (FP32 distance test, the point included): the
 *                    normals psulvsb_fpfh returns with normal_radius = radius, bit for bit, for any feature_radius <=
 *                    radius.
 *   3 <= max_nn <= 32: hybrid neighbourhood (Open3D's KDTreeSearchParamHybrid), the max_nn nearest points within
 *                    `radius`, ranked by (FP32 squared distance, index): ties go to the lower index.  A neighbourhood
 *                    of at most max_nn points gives the radius mode's normal bit for bit.
 * FP64 mean and covariance, smallest eigenvector, flipped towards the viewpoint (NULL: origin); fewer than 3 points:
 * NaN.  Results are bit-identical from call to call.  d_work: psulvsb_normals_workspace_bytes(n) bytes of device
 * scratch (depends on n only, never more than psulvsb_fpfh_workspace_bytes(n)).  PSULVSB_ERR_INVALID before any
 * device work for a radius that is not finite and > 0, another max_nn, a negative size or a required NULL; the batch
 * variants take the FPFH batch's items and return its errors, PSULVSB_ERR_UNSUPPORTED included.  n = 0 or B = 0 does
 * nothing.  Batch: cloud c's normals are rows [sum_{a<c} n_a, ...) of the (sum n) x 3 doubles, bit-identical to the
 * single call on cloud c alone (with its viewpoint).  The _host variants take host buffers and are synchronous. */
unsigned long long psulvsb_normals_workspace_bytes(int n);
int psulvsb_normals(void* stream, const double* d_pts, int n, double radius, int max_nn, const double viewpoint[3],
                    void* d_work, double* d_normals);
int psulvsb_normals_host(const double* pts, int n, double radius, int max_nn, const double viewpoint[3],
                         double* normals);
/* Device scratch of psulvsb_normals_batch (depends on the sizes only); 0 for B <= 0 or a negative size. */
unsigned long long psulvsb_normals_batch_workspace_bytes(const psulvsb_fpfh_cloud_t* clouds, int B);
int psulvsb_normals_batch(void* stream, const psulvsb_fpfh_cloud_t* clouds, int B, double radius, int max_nn,
                          void* d_work, double* d_normals);
int psulvsb_normals_batch_host(const psulvsb_fpfh_cloud_t* clouds, int B, double radius, int max_nn,
                               double* normals);

/* ---- Voxel downsampling (DESIGN.md section 10, "Voxel downsampling"): Open3D's PointCloud::VoxelDownSample on the
 * GPU.  Points and voxels are column-major 3xn doubles.  A point with a non-finite coordinate is dropped; lo = the
 * minimum of the finite points per coordinate, origin = lo - voxel_size * 0.5, and a point's cell is
 * floor((p - origin) / voxel_size) per coordinate in FP64, converted to int64 with saturation.  Two points share a
 * voxel iff their three cells are equal.  Each voxel gives the mean of its members (FP64 sums in ascending input
 * index, then one division by the count); voxels come out in ascending order of their lowest input index, so a cloud
 * with at most one point per voxel comes back in input order.  Results are bit-identical from call to call.
 * Capacity = input size: d_out holds 3 x n doubles, of which the first *d_count columns are voxels (the rest is
 * unspecified).  d_work: psulvsb_voxel_down_sample_workspace_bytes(n) bytes of device scratch (depends on n only; 0
 * for n < 0).  The device variants are asynchronous on `stream` and leave the count on the device.
 * PSULVSB_ERR_INVALID before any device work for a voxel_size that is not finite and > 0, a negative size, a NULL
 * points pointer of a non-empty cloud, a required NULL output or B < 0; PSULVSB_ERR_UNSUPPORTED when the sizes add up
 * to 2^31 or more (the FPFH batch's rule).  n = 0 or B = 0 does nothing beyond writing zero counts: the _host
 * variants write them on the host and need no device when every cloud is empty; the device variants write them on the
 * device, so an empty single call still needs one (B = 0 writes nothing and needs none).  Batch: items are
 * psulvsb_fpfh_cloud_t (the viewpoint is ignored); cloud c's voxels are columns [sum_{a<c} n_a, ... + counts[c]) of
 * the 3 x (sum n) doubles, bit-identical to the single call on cloud c alone.  The _host variants take host buffers
 * and are synchronous. */
unsigned long long psulvsb_voxel_down_sample_workspace_bytes(int n);
int psulvsb_voxel_down_sample(void* stream, const double* d_pts, int n, double voxel_size, void* d_work,
                              double* d_out /* 3 x n capacity */, int* d_count);
int psulvsb_voxel_down_sample_host(const double* pts, int n, double voxel_size, double* out /* 3 x n */, int* n_out);
/* Device scratch of psulvsb_voxel_down_sample_batch (depends on the sizes only); 0 for B <= 0 or a negative size. */
unsigned long long psulvsb_voxel_down_sample_batch_workspace_bytes(const psulvsb_fpfh_cloud_t* clouds, int B);
int psulvsb_voxel_down_sample_batch(void* stream, const psulvsb_fpfh_cloud_t* clouds, int B, double voxel_size,
                                    void* d_work, double* d_out, int* d_counts);
int psulvsb_voxel_down_sample_batch_host(const psulvsb_fpfh_cloud_t* clouds, int B, double voxel_size,
                                         double* out, int* counts);

typedef struct psulvsb_match_pair {
  const double* src;  /* 3 x n_src, column-major: the tuple test's points                                 */
  int n_src;
  const double* tgt;  /* 3 x n_tgt                                                                        */
  int n_tgt;
  const float* fs;    /* n_src x 33 descriptors                                                           */
  const float* ft;    /* n_tgt x 33                                                                       */
  uint64_t seed;      /* the tuple test's Philox key for this pair                                        */
} psulvsb_match_pair_t;
/* Output layout: pair b's (source, target) index pairs (interleaved ints) begin at pair offset sum_{a<b} cap_a with
 *   cap = 0 when a side is empty, else 3000 with the tuple test, else n_src with crosscheck and n_src + n_tgt without;
 * counts[b] receives pair b's count (at most cap_b).  Device scratch of psulvsb_match_batch (depends on the sizes and
 * the flags only); 0 for B <= 0 or a negative size. */
unsigned long long psulvsb_match_batch_workspace_bytes(const psulvsb_match_pair_t* pairs, int B, int crosscheck,
                                                       int tuple_test);
/* Asynchronous on `stream`, without a host round trip: d_pairs holds sum cap pairs, d_counts[B] long longs. */
int psulvsb_match_batch(void* stream, const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test,
                        double tuple_scale, void* d_work, int* d_pairs, long long* d_counts);
/* The same on host buffers, synchronous; pairs_out holds sum cap pairs (entries past counts[b] are unspecified). */
int psulvsb_match_batch_host(const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test,
                             double tuple_scale, int* pairs_out, long long* counts);

/* ---- Refinement of a registration on the raw clouds (DESIGN.md section 11): rigid ICP, point-to-point or
 * point-to-plane, in the loop of Open3D's registration_icp -- evaluate T0; then repeatedly compute the update U from
 * the current correspondences, set T <- U T and evaluate T; stop when both |d fitness| < relative_fitness and
 * |d inlier_rmse| < relative_rmse, or after max_iterations updates.  The correspondence of a source point (transformed
 * from the original P by T in FP64) is the target point at the smallest squared distance <= d^2 (ties: lowest index;
 * point-to-plane skips targets with a non-finite normal).  Convention q ~ R p + t; R column-major.  Every sum has one
 * fixed order, so results are bit-identical from call to call.  Parity with Open3D / PCL is unpinned; the tests compare
 * with a numpy restatement (oracle/icp.py). */
typedef struct psulvsb_icp_params {
  double max_correspondence_distance; /* d: finite, > 0                                                  */
  double relative_fitness;            /* >= 0 (default 1e-6)                                             */
  double relative_rmse;               /* >= 0 (default 1e-6)                                             */
  int max_iterations;                 /* updates at most (default 30); 0 = evaluate T0 only             */
  int point_to_plane;                 /* 0: point-to-point (Umeyama without scale), 1: point-to-plane   */
} psulvsb_icp_params_t;

enum {
  PSULVSB_ICP_CONVERGED = 0,     /* the relative rule stopped the loop                                  */
  PSULVSB_ICP_MAX_ITERATIONS = 1,/* max_iterations updates were applied                                 */
  PSULVSB_ICP_NO_UPDATE = 2      /* too few correspondences (< 3 point-to-point, < 6 point-to-plane), a non-positive
                                    pivot or a non-finite solution of the 6x6 system, or an empty cloud: T is the last
                                    transform evaluated                                                  */
};

typedef struct psulvsb_icp_result {
  double rotation[9]; /* column-major                                                                     */
  double translation[3];
  double fitness;     /* correspondences / n_s at the final T                                             */
  double inlier_rmse; /* sqrt(sum d^2 / correspondences), 0 without correspondences                        */
  int n_correspondences;
  int iterations;     /* updates applied                                                                   */
  int status;         /* PSULVSB_ICP_*                                                                     */
} psulvsb_icp_result_t;

/* Trace record k: the evaluation of T_k (k = 0 .. iterations). */
typedef struct psulvsb_icp_iteration {
  double rotation[9];
  double translation[3];
  double fitness;
  double inlier_rmse;
  int n_correspondences;
} psulvsb_icp_iteration_t;

/* max_correspondence_distance 0 (invalid: the caller sets it), max_iterations 30, relative criteria 1e-6,
 * point-to-point. */
void psulvsb_icp_default_params(psulvsb_icp_params_t* p);
/* Device scratch of psulvsb_icp (depends on the sizes only); 0 for a negative size. */
unsigned long long psulvsb_icp_workspace_bytes(int n_s, int n_t);
/* d_src 3 x n_s, d_tgt 3 x n_t, d_tgt_normals 3 x n_t (required for point-to-plane, else ignored): column-major
 * doubles on the device.  R0 (column-major) and t0 on the host.  Asynchronous on `stream`: no host round trip inside
 * the loop.  d_result: one psulvsb_icp_result_t on the device; d_trace (may be NULL): room for max_iterations + 1
 * records, of which iterations + 1 are written; d_corr (may be NULL): n_s ints, the target index of every source point
 * at the final T or -1.  An empty cloud returns T0 with fitness 0, 0 iterations and PSULVSB_ICP_NO_UPDATE.  Bad
 * arguments (negative sizes, a non-finite or non-positive d, max_iterations < 0, negative or NaN relative criteria,
 * point_to_plane not 0 / 1 or without normals, a required NULL, non-finite R0 / t0) return PSULVSB_ERR_INVALID before
 * any device work. */
int psulvsb_icp(void* stream, const double* d_src, int n_s, const double* d_tgt, int n_t, const double* d_tgt_normals,
                const psulvsb_icp_params_t* params, const double R0[9], const double t0[3], void* d_work,
                psulvsb_icp_result_t* d_result, psulvsb_icp_iteration_t* d_trace, int* d_corr);
/* The same on host buffers, synchronous (one device-to-host copy at the end). */
int psulvsb_icp_host(const double* src, int n_s, const double* tgt, int n_t, const double* tgt_normals,
                     const psulvsb_icp_params_t* params, const double R0[9], const double t0[3],
                     psulvsb_icp_result_t* result, psulvsb_icp_iteration_t* trace, int* corr);

/* ---- A batch of B independent ICP problems in one call (DESIGN.md section 11, "Batches"): every pair has its own
 * clouds, target normals and initial transform; all share one psulvsb_icp_params_t.  Every launch covers all pairs, so
 * a call issues as many launches as psulvsb_icp whatever B is.  Pair b's result, trace records and correspondences are
 * bit-identical to what psulvsb_icp_host returns for that pair alone (an empty cloud included). */
typedef struct psulvsb_icp_pair {
  const double* src;         /* 3 x n_s, column-major                                                  */
  int n_s;
  const double* tgt;         /* 3 x n_t                                                                */
  int n_t;
  const double* tgt_normals; /* 3 x n_t, point-to-plane only (else ignored)                            */
  double R0[9];              /* column-major                                                           */
  double t0[3];
} psulvsb_icp_pair_t;

/* Device scratch of psulvsb_icp_batch (depends on the pairs' sizes only); 0 for B <= 0 or a negative size. */
unsigned long long psulvsb_icp_batch_workspace_bytes(const psulvsb_icp_pair_t* pairs, int B);
/* pairs: a HOST array whose cloud pointers are device pointers; it is read before the call returns.  Asynchronous on
 * `stream`.  d_work: psulvsb_icp_batch_workspace_bytes(pairs, B) bytes; d_results[B]; d_trace (may be NULL):
 * B * (max_iterations + 1) records, pair b's from b * (max_iterations + 1); d_corr (may be NULL): sum of n_s ints, pair
 * b's from sum_{a<b} n_s(a), target indices local to the pair.  PSULVSB_ERR_INVALID before any device work for B < 0,
 * the parameters psulvsb_icp refuses, a required NULL, a pair with a negative size, a NULL cloud that is not empty, a
 * non-finite R0 / t0, or point-to-plane without normals on a pair with n_t > 0; PSULVSB_ERR_UNSUPPORTED when the
 * pairs' n_s or n_t add up to 2^31 or more.  B = 0 does nothing. */
int psulvsb_icp_batch(void* stream, const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                      void* d_work, psulvsb_icp_result_t* d_results, psulvsb_icp_iteration_t* d_trace, int* d_corr);
/* The same on host buffers (pairs' pointers are host pointers), synchronous: one upload of the clouds and one download
 * of results[B], trace (may be NULL; iterations + 1 records of pair b written from b * (max_iterations + 1)) and corr
 * (may be NULL). */
int psulvsb_icp_batch_host(const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                           psulvsb_icp_result_t* results, psulvsb_icp_iteration_t* trace, int* corr);

/* ---- Generalized ICP (plane-to-plane, Segal et al.; Open3D's registration_generalized_icp), DESIGN.md section 11
 * "Generalized ICP": the loop, stop rule, correspondences (every target point is a candidate), trace, results and
 * statuses of psulvsb_icp; only the update differs.  Each point's covariance is I - (1 - epsilon) n n^T for its unit
 * normal n (normalised in FP64; a non-finite or zero normal gives I); the update solves the Gauss-Newton system of
 * sum d^T (Sigma_t + R Sigma_s R^T)^-1 d with Open3D's Jacobian by the 6x6 Cholesky of point-to-plane, and needs 3
 * correspondences.  params->point_to_plane must be 0 (the entry point is the mode); epsilon: finite, 0 < epsilon <= 1
 * (Open3D's default 1e-3; 1 gives the linearised point-to-point step).  The sign of a normal does not matter.  The
 * tests compare with a numpy restatement (tests/gicp_restatement.py). */
typedef struct psulvsb_gicp_pair {
  const double* src;         /* 3 x n_s, column-major                                                  */
  int n_s;
  const double* tgt;         /* 3 x n_t                                                                */
  int n_t;
  const double* src_normals; /* 3 x n_s, required when n_s > 0 and n_t > 0                             */
  const double* tgt_normals; /* 3 x n_t, required when n_s > 0 and n_t > 0                             */
  double R0[9];              /* column-major                                                           */
  double t0[3];
} psulvsb_gicp_pair_t;

/* psulvsb_icp with generalized ICP's update.  Workspace: psulvsb_icp_workspace_bytes(n_s, n_t).  PSULVSB_ERR_INVALID
 * before any device work for every argument psulvsb_icp refuses, an epsilon outside (0, 1] or NaN, point_to_plane != 0,
 * or a NULL normal array when n_s > 0 and n_t > 0. */
int psulvsb_gicp(void* stream, const double* d_src, int n_s, const double* d_src_normals, const double* d_tgt, int n_t,
                 const double* d_tgt_normals, const psulvsb_icp_params_t* params, double epsilon, const double R0[9],
                 const double t0[3], void* d_work, psulvsb_icp_result_t* d_result, psulvsb_icp_iteration_t* d_trace,
                 int* d_corr);
/* The same on host buffers, synchronous: clouds and normals go up in one copy, one device-to-host copy at the end. */
int psulvsb_gicp_host(const double* src, int n_s, const double* src_normals, const double* tgt, int n_t,
                      const double* tgt_normals, const psulvsb_icp_params_t* params, double epsilon,
                      const double R0[9], const double t0[3], psulvsb_icp_result_t* result,
                      psulvsb_icp_iteration_t* trace, int* corr);
/* Device scratch of psulvsb_gicp_batch: psulvsb_icp_batch_workspace_bytes of the same sizes. */
unsigned long long psulvsb_gicp_batch_workspace_bytes(const psulvsb_gicp_pair_t* pairs, int B);
/* psulvsb_icp_batch with generalized ICP's update: the layouts, refusals and the guarantee that pair b's outputs are
 * bit-identical to psulvsb_gicp_host on that pair alone are psulvsb_icp_batch's, plus psulvsb_gicp's refusals. */
int psulvsb_gicp_batch(void* stream, const psulvsb_gicp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                       double epsilon, void* d_work, psulvsb_icp_result_t* d_results, psulvsb_icp_iteration_t* d_trace,
                       int* d_corr);
/* The same on host buffers, synchronous: one upload of the clouds and normals, one download (psulvsb_icp_batch_host). */
int psulvsb_gicp_batch_host(const psulvsb_gicp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                            double epsilon, psulvsb_icp_result_t* results, psulvsb_icp_iteration_t* trace, int* corr);

/* Clique escalation (registration.cc:1000-1085 -> teaser/src/graph.cc:12-125, PMC exact maximum clique) of the
 * graph with n_vertices vertices and the given edges (uint2 endpoint pairs).  A deterministic greedy maximal
 * clique (most neighbours among the remaining candidates first, ties: lowest index) gives the lower bound;
 * exact != 0 then runs a branch and bound from every vertex of sufficient degree (one warp per root, local
 * bit matrix in shared memory) and keeps the largest clique (ties: lowest root).
 * d_adj: scratch of psulvsb_max_clique_scratch_words(n_vertices) 32-bit words.  d_flags[n_vertices] (u8)
 * receives the membership, d_size[0] the clique size, d_size[1] = 1 when the size is proven maximum (0: a
 * neighbourhood above 512 vertices or the node budget stopped the search; the greedy answer stands).
 * Which maximum clique PMC returns is not unique: parity for this branch is defined on the size. */
unsigned long long psulvsb_max_clique_scratch_words(int n_vertices);
int psulvsb_max_clique(void* stream, const void* d_edges_uint2, unsigned long long n_edges, int n_vertices,
                       uint32_t* d_adj, uint8_t* d_flags, int* d_size, int exact);

/* Stage 4 -- fused transform + score + argmax (registration.cc:1303-1336, :1417-1444):
 * counts[h] = #{ j : | q_j - s (R_h p_j + t_h) | <= tau } over all n points, evaluated in FP32
 * from float4 tiles with every point inside the FP32 error band re-evaluated in FP64, plus the
 * argmax packed as (count << 32) | (0xFFFFFFFF - h) in *d_best (first best hypothesis wins).
 * *d_best is combined with atomicMax, not overwritten: zero it before the first call (calls over
 * parts of one hypothesis set with their hyp_begin may then share it).  d_best and
 * d_border_count (units re-evaluated in FP64, added to *d_border_count) may be NULL.
 * d_hyp: n_hyp x 12 doubles (R column-major then t).  hyp_begin offsets the ids written into
 * d_best (hypothesis sharding across GPUs); hyp_begin + n_hyp must not exceed 0xFFFFFFFF
 * (PSULVSB_ERR_UNSUPPORTED).  center_src / center_dst: the (host) centres the float4 tiles were
 * packed with (psulvsb_pack_points), NULL = 0; coord_bound: max |coordinate| of the packed tiles.
 * n = 0 zeroes the counts (and *d_best receives the first hypothesis's key); n < 0 is
 * PSULVSB_ERR_INVALID.  When tau^2 or the error band exceeds the FP32 range, every point is
 * re-evaluated in FP64: the counts stay exact, at FP64 speed. */
int psulvsb_score_batch(void* stream, const void* d_src_f4, const void* d_dst_f4, const double* d_src64,
                        const double* d_dst64, int n, const double* d_hyp, unsigned long long n_hyp,
                        unsigned long long hyp_begin, double scale, double tau, double coord_bound,
                        const double center_src[3], const double center_dst[3], uint32_t* d_counts,
                        unsigned long long* d_best, unsigned long long* d_border_count);
/* ------------------------------------------------------------------------------------------ */
/* multi-GPU: one process per GPU, one NCCL communicator per handle (SURVEY.md 8e).  The reference  */
/* is single-threaded CPU code and has no counterpart; the path shards where its work splits:       */
/* independent registrations (no exchange: give every rank its own slice of psulvsb_solve_batch),   */
/* hypothesis batches (psulvsb_score_batch_sharded) and, for one large registration, the rows of    */
/* the consistency stage (psulvsb_solve_sharded; loop registration.cc:682-767).                     */
/* ------------------------------------------------------------------------------------------ */
#define PSULVSB_UNIQUE_ID_BYTES 128
/* Rank 0 makes the communicator id (ncclGetUniqueId) and hands its PSULVSB_UNIQUE_ID_BYTES bytes to the other ranks by
 * any means it has (MPI, a socket, a file, torch.distributed); then every rank calls psulvsb_comm_create with its rank.
 * NCCL is bound at run time (libnccl.so.2); without it these entry points fail with PSULVSB_ERR_UNSUPPORTED. */
int psulvsb_comm_unique_id(void* out_id);
int psulvsb_comm_create(psulvsb_handle_t h, int rank, int world, const void* id);
int psulvsb_comm_destroy(psulvsb_handle_t h);
int psulvsb_comm_rank(psulvsb_handle_t h);
/* The row block [begin, end) of the consistency stage that psulvsb_solve_sharded gives rank `rank` of `world`: every
 * rank owns about the same number of line vectors (row i has n - 1 - i of them).  Host arithmetic, no device. */
int psulvsb_shard_row_range(int n, int rank, int world, int* begin, int* end);
int psulvsb_comm_world(psulvsb_handle_t h);
/* In-stream collectives on DEVICE buffers (no-ops on a handle without a communicator): element-wise sum of uint32
 * (per-row popcounts of row blocks built with psulvsb_consistency_mask_rows: rows a rank does not own stay 0, so the
 * sum is the all-gather) and max of uint64 (packed best-hypothesis keys). */
int psulvsb_comm_allreduce_sum_u32(psulvsb_handle_t h, void* stream, uint32_t* d_inout, unsigned long long n);
int psulvsb_comm_allreduce_max_u64(psulvsb_handle_t h, void* stream, unsigned long long* d_inout, unsigned long long n);
/* psulvsb_score_batch over this rank's slice of the hypotheses (hyp_begin = the slice's first global id) followed, on
 * the same stream, by ONE 8-byte ncclAllReduce(max) of *d_best: afterwards every rank holds the global best key. */
int psulvsb_score_batch_sharded(psulvsb_handle_t h, void* stream, const void* d_src_f4, const void* d_dst_f4,
                                const double* d_src64, const double* d_dst64, int n, const double* d_hyp,
                                unsigned long long n_hyp, unsigned long long hyp_begin, double scale, double tau,
                                double coord_bound, const double center_src[3], const double center_dst[3],
                                uint32_t* d_counts, unsigned long long* d_best, unsigned long long* d_border_count);
/* psulvsb_solve of ONE (large) registration by all ranks of the handle's communicator: every rank passes the SAME
 * problem and params and receives the same solution.  Rank r builds a triangular-balanced block of the consistency
 * mask's rows and compacts its edges; the ranks exchange their edge counts (8 bytes each) and then their blocks of the
 * edge list (in-place all-gather-v over NVLink), so that every rank holds the reference's L_reduced_set in the
 * reference's row-major order; the sequential RANSAC that follows is replicated (it is deterministic: same sample
 * stream, same result).  Known scale only.  Without a communicator (or world = 1) this is psulvsb_solve. */
int psulvsb_solve_sharded(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                          psulvsb_solution_t* solution, psulvsb_trace_t* trace /* may be NULL */);

/* Single-hypothesis FP64 scoring with per-point outputs (inlier flags, residuals). */
int psulvsb_score_one(void* stream, const double* d_src64, const double* d_dst64, int n, double scale,
                      const double* d_R, const double* d_t, double tau, uint8_t* d_inliers, double* d_residuals,
                      int* d_count);

#ifdef __cplusplus
}
#endif
#endif /* PSULVSB_H_ */
