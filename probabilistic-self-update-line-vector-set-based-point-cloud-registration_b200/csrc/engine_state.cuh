// engine_state.cuh -- device-resident per-registration state of the lock-step batch engine.
//
// The reference keeps this state in locals of solve() (registration.cc:622-1535) and in
// file-scope globals (registration.cc:36-50: first_time, *_last_best, scale_noise,
// translation_noise, longholi).  Here it is one POD per registration in HBM, read and written
// only by the control kernels (engine.cu), so B registrations advance together without the host.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "engine.cuh"

namespace psulvsb {

enum : int { PHASE_ROUND_START = 0, PHASE_LOCAL = 1, PHASE_DONE = 2,
             PHASE_HOST_SCORE = 3 };  // (split host scoring only: between the control kernel and the two kernels after it)

struct Xform {
  double s;
  double R[9];  // row-major
  double t[3];
};

// what reset(params_) + the in-loop overrides hand to the sub-solvers (registration.cc:937-945)
struct SubParams {
  double noise_bound, cbar2;
  int max_iterations;
  double gnc_factor, cost_threshold;
};

struct EngineParams {
  SubParams caller, inloop;
  int sampler_counters;      // sample_list_counters(): entries of JobCtl::bcount
  int zero_sampler_scratch;  // 1: engine_init_kernel clears the accept bitmask / value bitmap (see engine.cu)
  double pr_noise;          // 2 * score_noise_bound (registration.cc:36)
  double score_sigma;       // score_noise_bound: sigma of computeInlierProbability (registration.cc:1428)
  double rotation_similar;  // registration.cc:48
  int local_max_iter;       // registration.cc:49
  double tpro_host, tpro_local;
  int host_round_limit;
  double wallclock_cap_s;
  int self_update;
  int inlier_selection_mode;
  int max_local_iters;  // engine guard against the reference's non-terminating inputs
  int split_host_scoring;  // 1: the host scoring of all M points runs as a grid-wide kernel of its own (large M)
};

struct JobCtl {
  // ---- per-solve constants
  int C0, M, Ccap;
  double* src;  // working set, column-major 3 x Ccap (grows under self-update, registration.cc:800-806)
  double* dst;
  const double* src0;  // pristine reduced set 3 x C0
  const double* dst0;
  const double* ori_src;  // 3 x M
  const double* ori_dst;
  const int* keep_mask0;
  const int* reduce_map0;
  int* keep_mask;  // [M] working copies
  int* reduce_map;
  int* inlier_counter;  // [M]
  int* new_corr;        // [M]
  int* inlier_history;  // [M]
  int* final_inliers;   // [M]
  uint32_t* hs_bits;    // [2 * ceil(M / 32)] split host scoring: per-point decisions (new correspondence, inlier map)
  int hs_curr;          // split host scoring: inliers counted so far
  double* residual_history;  // [M]
  int* inlier_map;           // [Ccap]
  int* idx;                  // [Ccap] translation scratch
  double* xs;                // [3 * (Ccap + 1)]
  double* xs_sorted;         // [translation_sort_doubles(Ccap)] sorting scratch of the max-stabbing translation
  uint8_t* sampled_flags;    // [Ccap]
  uint8_t* rot_flags;        // [Ccap]
  void* edges;               // reduced set (L_reduced_set) as endpoint pairs, EdgeNarrow or EdgeWide (edge_fmt.cuh)
  unsigned long long edge_cap;
  uint32_t* vbits;            // sampler value bitmap of the L sample [ceil(edge_cap / 32)], zero between uses
  uint32_t* blist;            // sampler bucket lists [blist_cap]
  unsigned long long blist_cap;
  unsigned int* bcount;       // [sample_list_counters()] zero between uses
  uint32_t* first;  // [first_words] sampler accept bitmask (zero between uses)
  unsigned long long first_words;
  uint32_t* draws;  // sampler draw-value cache [draws_cap]
  unsigned long long draws_cap;
  unsigned long long* chunk_prefix;  // sampler scratch
  unsigned int* ticket;              // sampler scratch (zero between uses)
  uint32_t* L_sampled;
  uint32_t* basic_idx;
  uint2* basic_edges;
  double* weights;
  double* lv;  // GNC-TLS line-vector scratch, SoA [6][lv_cap]
  unsigned long long lv_cap;
  double* pts8;        // [Ccap][8] working points as 64-byte records (sx sy sz tx ty tz 0 0) for the GNC prologue
  uint32_t* gnc_perm;  // [2][lv_cap] index scratch of the GNC kernel's line-vector parking
  double* gnc_grid_red;        // grid mode of the GNC kernel (few registrations): partial results of its CTAs, or NULL
  unsigned int* gnc_grid_bar;  // ... and their arrival counter
  uint32_t* adj;        // clique escalation: Ccap x adj_stride bit matrix
  int adj_stride;
  uint8_t* clique_flags;  // [Ccap]
  uint2* pruned_edges;  // unknown scale: scale-inlier line vectors handed to the rotation solver
  int estimate_scaling;
  psulvsb_local_trace_t* local_trace;
  psulvsb_host_trace_t* host_trace;
  int local_trace_cap, host_trace_cap;
  uint64_t seed;
  double tau;  // PrNoise * (1 + (float)C0 / M)   (registration.cc:669, :1424)
  // ---- dynamic
  int C;
  unsigned long long n_red, n_red0, n_ls;
  int n_sampled_pts, basic_choose;
  int phase, status;
  int rounds_left, host_round, local_iter_global, host_scorings, escalations;
  int first_time, sampled_first_time, inloop, longholi, rate_idx;
  int local_r, host_r, best_sampled_cnt, best_host_cnt;
  double pro_local, pro_host;
  int pro_host_not_over;
  double scale_noise, translation_noise;
  Xform sol, best_sampled, best_host, last_best;
  int new_corr_count, inlier_map_size;
  int scale_calls, n_pruned;
  int clique_size, clique_proven, aborted;
  double cur_scale;  // solution_.scale of the iteration in flight (registration.cc:958-991)
  unsigned long long sample_status[2];
  double R_gnc[9];  // column-major (GncJob::R_out)
  int gnc_info[4];
  double gnc_cost;
  SubParams cur;  // parameters of the local iteration in flight
  int n_local_trace, n_host_trace;
  int valid, refined;
};

}  // namespace psulvsb
