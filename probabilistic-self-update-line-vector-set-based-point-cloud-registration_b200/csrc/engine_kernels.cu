// engine_kernels.cu -- control kernels of the lock-step batch engine: the two-level RANSAC state
// machine of RobustRegistrationSolver::solve (registration.cc:783-1488) and the final refinement
// (registration.cc:1499-1525), one CTA per registration, no host round trip.
//
// One engine "tick" = one local iteration (registration.cc:903-1488) of every unfinished
// registration:  round_start -> [L sample] -> [basic sample] -> GNC-TLS -> local_control.
// The stage kernels in between read device-resident job descriptors that these kernels rewrite.
#include <cuda_runtime.h>

#include "common.cuh"
#include "engine.cuh"
#include "engine_kernels.cuh"
#include "engine_state.cuh"
#include "solve_dev.cuh"
#include "svd3.cuh"

namespace psulvsb {

static_assert(kCtlThreads == BLK, "control kernels assume BLK threads");

namespace {

__device__ __constant__ double kLRate[4] = {0.1, 0.2, 0.5, 1.0};  // registration.cc:776, :1377-1388
__device__ __constant__ double kBRate[4] = {0.3, 0.3, 0.3, 1.0};  // registration.cc:777

__device__ __forceinline__ void xform_identity(Xform& x) {
  x.s = 1.0;
#pragma unroll
  for (int i = 0; i < 9; ++i) x.R[i] = (i % 4 == 0) ? 1.0 : 0.0;
  x.t[0] = x.t[1] = x.t[2] = 0.0;
}

// 1 - gamma_p(3/2, z), z = r^2 / (2 sigma^2)  (computeInlierProbability, registration.cc:611-619;
// closed form of Boost's gamma_p(1.5, z))
__device__ __forceinline__ double inlier_probability(double r, double sigma) {
  const double z = (r * r) / (2.0 * sigma * sigma);
  if (!(z > 0)) return 1.0;
  return erfc(sqrt(z)) + 2.0 * sqrt(z / 3.14159265358979323846) * exp(-z);
}

// Prepares the basic-subset draw (registration.cc:908-933) and the rotation solve
// (registration.cc:1102-1111) of the next local iteration.  Thread 0 only.
__device__ void prepare_local(JobCtl& J, SampleJob& sb, GncJob& g, CliqueJob& q, const EngineParams& P) {
  const double b_rate = kBRate[J.rate_idx];
  J.basic_choose = (int)((double)J.n_ls * b_rate);
  // reset(params_) then the overrides: THIS iteration sees the previous contents (SURVEY defect 6)
  J.cur = J.inloop ? P.inloop : P.caller;
  J.inloop = 1;
  sb.seed = J.seed;
  sb.domain = PSULVSB_DOMAIN_BASIC;
  sb.event = (uint32_t)J.local_iter_global;
  sb.n = J.n_ls;
  sb.count = (unsigned long long)J.basic_choose;
  sb.max_draws = sample_max_draws_formula(sb.n, sb.count);
  sb.first = J.first;
  sb.chunk_prefix = J.chunk_prefix;
  sb.ticket = J.ticket;
  sb.draws = J.draws;
  sb.draws_cap = J.draws_cap;
  sb.blist = J.blist;
  sb.blist_cap = J.blist_cap;
  sb.bcount = J.bcount;
  sb.out = J.basic_idx;
  sb.status = &J.sample_status[1];
  sb.identity = 0;
  sb.post = 2;
  sb.vbits = nullptr;
  sb.edges = J.edges;
  sb.via = J.L_sampled;
  sb.gathered = J.basic_edges;
  sb.pts8 = J.pts8;
  sb.lv_out = J.estimate_scaling ? nullptr : J.lv;  // known scale: the emit pass forms the GNC-TLS line vectors
  sb.lv_cap = J.lv_cap;
  sb.flags = nullptr;
  sb.n_points = 0;
  sb.active = (J.basic_choose > 0) ? 1 : 0;
  J.sample_status[1] = 1ull;
  const double scale = 1.0;  // known scale (registration.cc:984-991)
  g.src = J.src;
  g.dst = J.dst;
  g.edges = J.basic_edges;
  g.K = (unsigned long long)J.basic_choose;
  g.inv_scale = 1.0 / scale;
  g.noise_bound = J.cur.noise_bound * (2.0 / scale);
  g.gnc_factor = J.cur.gnc_factor;
  g.cost_threshold = J.cur.cost_threshold;
  g.max_iterations = J.cur.max_iterations;
  g.use_init = J.first_time ? 0 : 1;
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int r = 0; r < 3; ++r) g.R_init[c * 3 + r] = J.last_best.R[r * 3 + c];
  g.weights = J.weights;
  g.lv = J.lv;
  g.lv_cap = J.lv_cap;
  g.perm = J.gnc_perm;
  g.grid_red = J.gnc_grid_red;
  g.grid_bar = J.gnc_grid_bar;
  g.pts8 = J.pts8;
  g.lv_ready = (J.estimate_scaling || sb.identity) ? 0 : 1;  // (unknown scale: pruned subset, rescaled -- formed in the kernel)
  g.R_out = J.R_gnc;
  g.inliers = nullptr;
  g.point_flags = J.rot_flags;
  g.n_points = J.C;
  g.info = J.gnc_info;
  g.prof = nullptr;
  g.cost = &J.gnc_cost;
  g.active = 1;
  // max-clique escalation (registration.cc:1000-1085): inlier graph of the round's scale-consistent line vectors
  q.active = (J.rate_idx == 3 && P.inlier_selection_mode != 3) ? 1 : 0;
  q.edges = J.basic_edges;
  q.n_edges = (unsigned long long)J.basic_choose;
  q.src = J.src;
  q.dst = J.dst;
  q.beta = 2.0 * J.cur.noise_bound * sqrt(J.cur.cbar2);  // ScaleInliersSelector with this iteration's params (:984-991)
  q.filter = 1;
  q.n_vertices = J.C;
  q.adj = J.adj;
  q.stride = J.adj_stride;
  q.flags = J.clique_flags;
  q.size = &J.clique_size;
  q.proven = &J.clique_proven;
}

// count_j [ | q_j - s (R p_j + t) | <= tau ] over the flagged points of the working set
__device__ int count_flagged(BlockScratch* s, const JobCtl& J, const Xform& X) {
  int cnt = 0, dummy = 0;
  for (int j = threadIdx.x; j < J.C; j += BLK)
    if (J.sampled_flags[j] && residual_ref(J.src + 3 * (size_t)j, J.dst + 3 * (size_t)j, X.s, X.R, X.t) <= J.tau) ++cnt;
  block_sum_int2(s, cnt, dummy);
  return cnt;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// init: working copies and dynamic state (the locals declared at registration.cc:655-680, :769-782)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLK)
    engine_init_kernel(JobCtl* __restrict__ jobs, SampleJob* __restrict__ sl, SampleJob* __restrict__ sb,
                       GncJob* __restrict__ gj, CliqueJob* __restrict__ cq,
                       const unsigned long long* __restrict__ n_edges, EngineParams P,
                       int* __restrict__ n_done) {
  JobCtl& J = jobs[blockIdx.x];
  // grid.y CTAs share a job's copies (one registration of 10^5 points alone: 12 MB through one SM took 0.8 ms); the
  // scalar state is thread 0's of the job's first CTA.  Nothing here reads what that thread writes.
  const int tid = blockIdx.y * BLK + threadIdx.x;
  const int stride = gridDim.y * BLK;
  for (int i = tid; i < 3 * J.C0; i += stride) {
    J.src[i] = J.src0[i];
    J.dst[i] = J.dst0[i];
  }
  // 64-byte point records (sx sy sz tx ty tz 0 0): the GNC prologue forms each line vector from two of them with
  // six 16-byte loads instead of twelve scattered 8-byte ones
  for (int i = tid; i < J.C0; i += stride) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      J.pts8[8 * (size_t)i + r] = J.src0[3 * (size_t)i + r];
      J.pts8[8 * (size_t)i + 3 + r] = J.dst0[3 * (size_t)i + r];
    }
    J.pts8[8 * (size_t)i + 6] = 0.0;
    J.pts8[8 * (size_t)i + 7] = 0.0;
  }
  for (int j = tid; j < J.M; j += stride) {
    J.keep_mask[j] = J.keep_mask0[j];
    J.reduce_map[j] = J.reduce_map0[j];
    J.inlier_counter[j] = 0;
    J.new_corr[j] = 0;
    J.inlier_history[j] = -1;
    J.final_inliers[j] = 0;
    J.residual_history[j] = 0.0;
  }
  // sampler scratch that every use leaves zeroed: only cleared when the host cannot vouch for it (first solve on this
  // arena layout, or the previous solve did not complete)
  if (P.zero_sampler_scratch)
    for (unsigned long long i = tid; i < J.first_words; i += stride) J.first[i] = 0u;  // sampler accept bitmask
  if (J.bcount)
    for (int i = tid; i < P.sampler_counters; i += stride) J.bcount[i] = 0u;  // sampler list counters
  if (P.zero_sampler_scratch)
    for (unsigned long long i = tid; i < (J.edge_cap + 31) / 32 + 32; i += stride) J.vbits[i] = 0u;
  if (tid == 0) {
    *J.ticket = 0u;
    J.C = J.C0;
    J.n_red0 = n_edges[blockIdx.x];
    J.n_red = J.n_red0;
    J.n_ls = 0;
    J.n_sampled_pts = 0;
    J.basic_choose = 0;
    J.phase = PHASE_ROUND_START;
    J.status = PSULVSB_OK;
    J.rounds_left = P.host_round_limit;
    J.host_round = 0;
    J.local_iter_global = 0;
    J.host_scorings = 0;
    J.escalations = 0;
    J.first_time = 1;
    J.sampled_first_time = 1;
    J.inloop = 0;
    J.longholi = 0;
    J.rate_idx = 0;
    J.local_r = 0;
    J.host_r = 0;
    J.best_sampled_cnt = 0;
    J.best_host_cnt = 0;
    J.pro_local = 0.0;
    J.pro_host = 0.0;
    J.pro_host_not_over = 1;
    J.scale_noise = 0.0;
    J.translation_noise = 0.0;
    xform_identity(J.sol);
    xform_identity(J.best_sampled);
    xform_identity(J.best_host);
    xform_identity(J.last_best);
    J.new_corr_count = 0;
    J.inlier_map_size = 0;
    J.scale_calls = 0;
    J.n_pruned = 0;
    J.cur_scale = 1.0;
    J.sample_status[0] = J.sample_status[1] = 1ull;
    J.n_local_trace = 0;
    J.n_host_trace = 0;
    J.valid = 0;
    J.refined = 0;
    sl[blockIdx.x].active = 0;
    sb[blockIdx.x].active = 0;
    gj[blockIdx.x].active = 0;
    cq[blockIdx.x].active = 0;
    J.clique_size = 0;
    J.aborted = 0;
    if (J.n_red0 > J.edge_cap) {
      J.status = PSULVSB_ERR_CAPACITY;
      J.phase = PHASE_DONE;
      atomicAdd(n_done, 1);
    } else if (J.n_red0 == 0) {
      // the reference never terminates here (p_local = NaN, registration.cc:1352/:1399): report invalid
      J.phase = PHASE_DONE;
      atomicAdd(n_done, 1);
    } else {
      atomicAdd(n_done + 1, 1);  // n_done[1]: registrations waiting for a round start
    }
  }
}

// ------------------------------------------------------------------------------------------
// round start: self-update append (registration.cc:786-832) and the L-sampled draw set-up
// (registration.cc:837-863)
// ------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(BLK)
    engine_round_start_kernel(JobCtl* __restrict__ jobs, SampleJob* __restrict__ sl, SampleJob* __restrict__ sb,
                              GncJob* __restrict__ gj, CliqueJob* __restrict__ cq, EngineParams P,
                              int* __restrict__ n_done) {
  JobCtl& J = jobs[blockIdx.x];
  SampleJob& L = sl[blockIdx.x];
  const int tid = threadIdx.x;
  if (J.phase != PHASE_ROUND_START) {
    if (tid == 0) {
      L.active = 0;
      if (J.phase == PHASE_DONE) {
        sb[blockIdx.x].active = 0;
        gj[blockIdx.x].active = 0;
        cq[blockIdx.x].active = 0;
      }
    }
    return;
  }
  __shared__ int ok_s;
  if (tid == 0) atomicSub(n_done + 1, 1);
  const int nnew = (P.self_update ? J.new_corr_count : 0);
  const int m0 = J.inlier_map_size;
  const int C = J.C;
  if (tid == 0) {
    const unsigned long long extra = (unsigned long long)nnew * (unsigned long long)m0 +
                                     (unsigned long long)nnew * (unsigned long long)(nnew > 0 ? nnew - 1 : 0) / 2ull;
    ok_s = (J.n_red + extra <= J.edge_cap && C + nnew <= J.Ccap) ? 1 : 0;
  }
  __syncthreads();
  if (!ok_s) {
    if (tid == 0) {
      J.status = PSULVSB_ERR_CAPACITY;
      J.phase = PHASE_DONE;
      L.active = 0;
      sb[blockIdx.x].active = 0;
      gj[blockIdx.x].active = 0;
      atomicAdd(n_done, 1);
    }
    return;
  }
  if (nnew > 0) {
    // points (registration.cc:800-806) and bookkeeping (:828-830)
    for (int i = tid; i < nnew; i += BLK) {
      const int o = J.new_corr[i];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        J.src[3 * (size_t)(C + i) + r] = J.ori_src[3 * (size_t)o + r];
        J.dst[3 * (size_t)(C + i) + r] = J.ori_dst[3 * (size_t)o + r];
        J.pts8[8 * (size_t)(C + i) + r] = J.ori_src[3 * (size_t)o + r];
        J.pts8[8 * (size_t)(C + i) + 3 + r] = J.ori_dst[3 * (size_t)o + r];
      }
      J.pts8[8 * (size_t)(C + i) + 6] = 0.0;
      J.pts8[8 * (size_t)(C + i) + 7] = 0.0;
      J.keep_mask[o] = 1;
      J.reduce_map[o] = C + i;
    }
    // line vectors new x (current inliers + earlier new ones), oriented (new, inlier) (:808-827)
    const unsigned long long base = J.n_red;
    for (int i = 0; i < nnew; ++i) {
      const unsigned long long off = base + (unsigned long long)i * m0 + (unsigned long long)i * (i > 0 ? i - 1 : 0) / 2ull;
      const int cnt = m0 + i;
      for (int j = tid; j < cnt; j += BLK) {
        const int other = (j < m0) ? J.inlier_map[j] : (C + (j - m0));
        F::store(J.edges, off + j, (unsigned)(C + i), (unsigned)other);
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    if (nnew > 0) {
      J.n_red += (unsigned long long)nnew * m0 + (unsigned long long)nnew * (nnew - 1) / 2ull;
      J.C = C + nnew;
    }
    J.rounds_left -= 1;
    J.new_corr_count = 0;
    J.inlier_map_size = 0;
    J.sampled_first_time = 1;
    J.best_sampled_cnt = 0;
    J.local_r = 0;
    J.pro_local = 0.0;
    const double l_rate = kLRate[J.rate_idx];
    unsigned long long n_ls = (unsigned long long)floor((double)J.n_red * l_rate);
    L.identity = 0;
    if (n_ls == 0) {  // registration.cc:839-847
      n_ls = J.n_red;
      L.identity = 1;
    }
    J.n_ls = n_ls;
    L.seed = J.seed;
    L.domain = PSULVSB_DOMAIN_L_SAMPLED;
    L.event = (uint32_t)J.host_round;
    L.n = J.n_red;
    L.count = n_ls;
    L.max_draws = L.identity ? 0ull : sample_max_draws_formula(L.n, L.count);
    L.first = J.first;
    L.chunk_prefix = J.chunk_prefix;
    L.ticket = J.ticket;
    L.draws = J.draws;
    L.draws_cap = J.draws_cap;
    L.blist = J.blist;
    L.blist_cap = J.blist_cap;
    L.bcount = J.bcount;
    L.out = J.L_sampled;
    L.status = &J.sample_status[0];
    L.post = 1;
    L.vbits = J.vbits;
    L.edges = J.edges;
    L.via = nullptr;
    L.gathered = nullptr;
    L.flags = J.sampled_flags;
    L.n_points = J.C;
    L.active = 1;
    J.sample_status[0] = 1ull;
    J.phase = PHASE_LOCAL;
    prepare_local(J, sb[blockIdx.x], gj[blockIdx.x], cq[blockIdx.x], P);
  }
}

int launch_round_start(cudaStream_t st, int n_jobs, JobCtl* jobs, SampleJob* sl, SampleJob* sb, GncJob* gj, CliqueJob* cq,
                       const EngineParams& P, int* n_done, bool narrow) {
  if (narrow)
    engine_round_start_kernel<EdgeNarrow><<<n_jobs, BLK, 0, st>>>(jobs, sl, sb, gj, cq, P, n_done);
  else
    engine_round_start_kernel<EdgeWide><<<n_jobs, BLK, 0, st>>>(jobs, sl, sb, gj, cq, P, n_done);
  PSU_CHECK_LAUNCH("engine_round_start_kernel");
  return PSULVSB_OK;
}

// ------------------------------------------------------------------------------------------
// unknown scale only: TLSScaleSolver on the basic subset (registration.cc:958-983 -> :397-415 ->
// ScalarTLSEstimator::estimate, scale branch, :66-120), pruning to the scale inliers, and the
// rotation-solve set-up that depends on the scale (registration.cc:1102-1108)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLK)
    engine_scale_kernel(JobCtl* __restrict__ jobs, GncJob* __restrict__ gj, CliqueJob* __restrict__ cq, EngineParams P) {
  JobCtl& J = jobs[blockIdx.x];
  if (J.phase != PHASE_LOCAL || !J.estimate_scaling) return;
  __shared__ BlockScratch scratch;
  __shared__ double est_s, scale_s;
  __shared__ int base_s;
  const int tid = threadIdx.x;
  const int K = J.basic_choose;
  const uint2* __restrict__ edges = J.basic_edges;
  double* __restrict__ X = J.weights;  // both arrays are dead again before the rotation solve starts
  double* __restrict__ A = J.lv;
  const double beta = 2.0 * J.cur.noise_bound * sqrt(J.cur.cbar2);
  double scale = J.cur_scale;
  int n_pruned = 0;
  if (K > 0) {
    for (int i = tid; i < K; i += BLK) {
      const uint2 e = edges[i];
      const double* sa = J.src + 3 * (size_t)e.x;
      const double* sb = J.src + 3 * (size_t)e.y;
      const double* ta = J.dst + 3 * (size_t)e.x;
      const double* tb = J.dst + 3 * (size_t)e.y;
      const double v1 = sqrt(sqnorm3(dsub(sb[0], sa[0]), dsub(sb[1], sa[1]), dsub(sb[2], sa[2])));
      const double v2 = sqrt(sqnorm3(dsub(tb[0], ta[0]), dsub(tb[1], ta[1]), dsub(tb[2], ta[2])));
      X[i] = v2 / v1;
      A[i] = dmul(beta, 1.0 / v1);
    }
    block_tls_scale(&scratch, X, A, K, J.seed, (uint32_t)J.scale_calls, !J.first_time, J.last_best.s, scale, &est_s,
                    &scale_s);
    const double est = est_s;
    scale = scale_s;
    // pruning (registration.cc:966-983): the consensus set of the UNREFINED estimate, in order
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int i0 = 0; i0 < K; i0 += BLK) {
      const int i = i0 + tid;
      const int f = (i < K && fabs(dsub(X[i], est)) <= A[i]) ? 1 : 0;
      int ea, eb, ta, tb;
      block_scan2(&scratch, f, 0, ea, eb, ta, tb);
      const int base = base_s;
      if (f) J.pruned_edges[base + ea] = edges[i];
      __syncthreads();
      if (tid == 0) base_s = base + ta;
      __syncthreads();
    }
    n_pruned = base_s;
  }
  __syncthreads();
  if (tid == 0) {
    if (K > 0) J.scale_calls += 1;
    J.scale_noise = beta;  // registration.cc:411
    J.cur_scale = scale;
    J.n_pruned = n_pruned;
    GncJob& g = gj[blockIdx.x];
    g.edges = J.pruned_edges;
    g.K = (unsigned long long)n_pruned;
    g.inv_scale = 1.0 / scale;                          // registration.cc:1102
    g.noise_bound = J.cur.noise_bound * (2.0 / scale);  // registration.cc:1106-1108
    CliqueJob& q = cq[blockIdx.x];  // the inlier graph uses the TLS scale inliers as they are (:1005-1012)
    q.edges = J.pruned_edges;
    q.n_edges = (unsigned long long)n_pruned;
    q.filter = 0;
  }
}

// ------------------------------------------------------------------------------------------
// local control: everything of one local iteration after the rotation solve
// (registration.cc:1114-1488)
// ------------------------------------------------------------------------------------------
// host scoring of ONE of the M correspondences (registration.cc:1417-1444): residual, inlier counter, self-update
// decision (add), inlier map entry (imap), histories.  Independent per point.
__device__ __forceinline__ void host_score_point(JobCtl& J, const EngineParams& P, const Xform& X, const uint32_t ev,
                                                 const int j, int& add, int& imap, int& inl) {
    const double res = residual_ref(J.ori_src + 3 * (size_t)j, J.ori_dst + 3 * (size_t)j, X.s, X.R, X.t);
    if (res <= J.tau) {
      inl = 1;
      J.inlier_counter[j] += 1;
      const int km = J.keep_mask[j];
      if (km == 0) {
        const int hst = J.inlier_history[j];
        if (hst == -1 || hst == 1)
          add = 1;
        else if (hst == 0)
          add = (philox_uniform01(J.seed, PSULVSB_DOMAIN_UNIFORM, ev, (uint64_t)j) <=
                 inlier_probability(res, P.score_sigma))
                    ? 1
                    : 0;
      }
      if (add) {
        J.final_inliers[j] = 1;
      } else if (km == 1) {
        imap = 1;
        J.final_inliers[j] = 1;
      }
      J.inlier_history[j] = 1;
    } else {
      // registration.cc:1438 (assignment-in-condition, SURVEY defect 2): the draw decides whether the
      // point's final_inliers flag is cleared; history := 0
      const double u = philox_uniform01(J.seed, PSULVSB_DOMAIN_UNIFORM, ev, (uint64_t)j);
      if (u > inlier_probability(J.residual_history[j], P.score_sigma)) J.final_inliers[j] = 0;
      J.inlier_history[j] = 0;
    }
    J.residual_history[j] = res;
}

// the end of a host round (registration.cc:1454-1488): best-host update, p_host, stop rules, next phase.  One thread.
__device__ void finish_host_round(JobCtl& J, const EngineParams& P, const Xform& X, const int curr, const double elapsed_s,
                                  SampleJob& sbj, GncJob& gjj, CliqueJob& cqj, int* __restrict__ n_done,
                                  const int new_corr_count, const int inlier_map_size) {
  const int M = J.M;
  J.host_r += J.local_r;
  J.host_scorings += 1;
  J.new_corr_count = new_corr_count;
  J.inlier_map_size = inlier_map_size;
  // the reference tests the already-escalated rate here (registration.cc:1454), not the one in
  // force when the iteration started
  const double b_now = kBRate[J.rate_idx];
  if (curr > J.best_host_cnt || J.pro_host == 0.0 || (b_now == 1.0 && curr >= J.best_host_cnt)) {
    J.best_host = X;
    J.best_host_cnt = curr;
  }
  J.last_best = J.best_host;
  J.pro_host = 1.0 - pow(1.0 - (double)((double)J.best_host_cnt / (double)M), J.host_r);
  const bool timeup = P.wallclock_cap_s > 0.0 && elapsed_s > P.wallclock_cap_s;
  if (J.pro_host > P.tpro_host || J.longholi || timeup) J.pro_host_not_over = 0;
  if (kLRate[J.rate_idx] == 1.0 && b_now == 1.0) J.longholi = 1;
  if (J.host_trace && J.n_host_trace < J.host_trace_cap) {
    psulvsb_host_trace_t& T = J.host_trace[J.n_host_trace++];
    T.host_round = J.host_round;
    T.curr_count = curr;
    T.best_host = J.best_host_cnt;
    T.new_corr_count = P.self_update ? J.new_corr_count : 0;
    T.inlier_map_size = J.inlier_map_size;
    T.host_r = J.host_r;
    T.p_host = J.pro_host;
  }
  J.host_round += 1;
  sbj.active = 0;
  gjj.active = 0;
  cqj.active = 0;
  if (J.pro_host_not_over && J.rounds_left > 0) {
    J.phase = PHASE_ROUND_START;
    atomicAdd(n_done + 1, 1);
  } else {
    J.valid = 1;
    J.phase = PHASE_DONE;
    atomicAdd(n_done, 1);
  }
}

__global__ void __launch_bounds__(BLK)
    engine_local_control_kernel(JobCtl* __restrict__ jobs, SampleJob* __restrict__ sl, SampleJob* __restrict__ sb,
                                GncJob* __restrict__ gj, CliqueJob* __restrict__ cq, EngineParams P, double elapsed_s,
                                int* __restrict__ n_done) {
  JobCtl& J = jobs[blockIdx.x];
  if (J.phase != PHASE_LOCAL) return;
  __shared__ BlockScratch scratch;
  __shared__ int base_s[2];
  __shared__ int similar_s;
  __shared__ Xform sol_s;
  const int tid = threadIdx.x;
  const int C = J.C;
  const double b_rate = kBRate[J.rate_idx];
  const bool clique_round = (b_rate == 1.0);

  const bool use_clique = clique_round && P.inlier_selection_mode != 3;
  if (J.sample_status[0] == 0ull || J.sample_status[1] == 0ull || (use_clique && J.clique_size <= 1)) {
    // sampler budget exhausted (never observed: mean + 8 sigma), or the inlier graph has no clique of
    // two vertices: the reference gives up there with valid = false (registration.cc:1032-1036)
    if (tid == 0) {
      if (J.sample_status[0] == 0ull || J.sample_status[1] == 0ull)
        J.status = PSULVSB_ERR_INTERNAL;
      else
        J.aborted = 1;
      J.phase = PHASE_DONE;
      sb[blockIdx.x].active = 0;
      gj[blockIdx.x].active = 0;
      cq[blockIdx.x].active = 0;
      atomicAdd(n_done, 1);
    }
    return;
  }

  // ---- |src_sampled| (registration.cc:870-894): the sampler leaves the endpoint set as flags
  if (J.sampled_first_time) {
    int c = 0, dummy = 0;
    for (int j = tid; j < C; j += BLK) c += J.sampled_flags[j] ? 1 : 0;
    block_sum_int2(&scratch, c, dummy);
    if (tid == 0) J.n_sampled_pts = c;
    __syncthreads();
  }

  // ---- rotation result (column-major) -> row-major
  if (tid == 0) {
    sol_s.s = J.cur_scale;
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) sol_s.R[r * 3 + c] = J.R_gnc[c * 3 + r];
    for (int r = 0; r < 3; ++r) sol_s.t[r] = J.sol.t[r];  // estimate starts from the previous value
    base_s[0] = 0;
  }
  __syncthreads();

  // ---- points handed to the translation solver: unique endpoints of the rotation inliers
  // (registration.cc:1114-1155), or every point in the max-clique round with selection NONE (:1066-1084)
  // (each thread takes a contiguous slice: one block scan for the whole set instead of one per 1024 points -- at
  // C = 100 000 the 98 scans were a quarter of this kernel; ascending j either way)
  {
    auto flagged = [&](int j) -> bool {
      // clique round: the clique's points (registration.cc:1238-1244); selection NONE: every point (:1066-1084)
      return clique_round ? (use_clique ? J.clique_flags[j] != 0 : true) : J.rot_flags[j] != 0;
    };
    const int per = (C + BLK - 1) / BLK;
    const int lo = min(C, tid * per), hi = min(C, lo + per);
    int c = 0;
    for (int j = lo; j < hi; ++j) c += flagged(j) ? 1 : 0;
    int ea, eb, ta, tb;
    block_scan2(&scratch, c, 0, ea, eb, ta, tb);
    int pos = ea;
    for (int j = lo; j < hi; ++j)
      if (flagged(j)) J.idx[pos++] = j;
    if (tid == 0) base_s[0] = ta;
    __syncthreads();
  }
  const int n_rot_pts = base_s[0];

  // ---- translation (registration.cc:1248-1250)
  {
    double t[3] = {sol_s.t[0], sol_s.t[1], sol_s.t[2]};
    double lb[3] = {J.last_best.t[0], J.last_best.t[1], J.last_best.t[2]};
    const double sigma = J.cur.noise_bound * sqrt(J.cur.cbar2);
    block_translation(&scratch, J.src, J.dst, J.idx, n_rot_pts, sol_s.s, sol_s.R, sigma, J.first_time ? nullptr : lb,
                      J.xs, t, J.xs_sorted);
    __syncthreads();
    if (tid == 0) {
      J.translation_noise = sigma;
      for (int r = 0; r < 3; ++r) sol_s.t[r] = t[r] / sol_s.s;
    }
  }
  __syncthreads();

  // ---- similarity with the last best (registration.cc:1261-1264)
  if (tid == 0) {
    int similar = 0;
    if (!J.first_time) {
      double tr = 0.0;
      for (int i = 0; i < 3; ++i) {
        // (R_last^T R)(i,i) = sum_k R_last(k,i) R(k,i)
        tr += (J.last_best.R[0 * 3 + i] * sol_s.R[0 * 3 + i] + J.last_best.R[1 * 3 + i] * sol_s.R[1 * 3 + i]) +
              J.last_best.R[2 * 3 + i] * sol_s.R[2 * 3 + i];
      }
      const double ang = fabs(acos(fmin(fmax((tr - 1.0) / 2.0, -1.0), 1.0)));
      const double d0 = J.last_best.t[0] - sol_s.t[0], d1 = J.last_best.t[1] - sol_s.t[1],
                   d2 = J.last_best.t[2] - sol_s.t[2];
      const double dn = sqrt((d0 * d0 + d1 * d1) + d2 * d2);
      similar = (fabs(J.last_best.s - sol_s.s) <= J.scale_noise && ang <= P.rotation_similar &&
                 dn <= J.translation_noise)
                    ? 1
                    : 0;
    }
    similar_s = similar;
  }
  __syncthreads();
  const int similar = similar_s;
  int curr_count = -1;
  if (!similar) {
    // registration.cc:1283-1345
    int last_cnt = -1;
    if (!J.first_time && b_rate < 1.0) last_cnt = count_flagged(&scratch, J, J.last_best);
    curr_count = count_flagged(&scratch, J, sol_s);
    if (tid == 0) {
      J.local_r += 1;
      if (last_cnt >= 0) {
        J.best_sampled_cnt = last_cnt;
        J.best_sampled = J.last_best;
      }
      if (curr_count > J.best_sampled_cnt || J.first_time) {
        J.best_sampled = sol_s;
        J.best_sampled_cnt = curr_count;
      }
      J.last_best = J.best_sampled;
      J.pro_local = 1.0 - pow(1.0 - (double)((double)J.best_sampled_cnt / (double)J.n_sampled_pts), J.local_r);
      J.first_time = 0;
      if ((J.local_r >= P.local_max_iter && J.pro_local <= 0.2) || b_rate == 1.0) {  // registration.cc:1361-1396
        J.pro_local = 1.0;
        if (J.rate_idx < 3) {
          J.rate_idx += 1;
          J.escalations += 1;
          if (J.rate_idx == 3) atomicAdd(n_done + 2, 1);  // n_done[2]: jobs that reached the clique round
        }
      }
    }
  } else if (tid == 0) {
    // registration.cc:1266-1281
    J.local_r += J.sampled_first_time ? (J.host_r + 1) : 1;
    J.pro_local = 1.0;
    J.best_sampled = sol_s;
  }
  __syncthreads();
  if (tid == 0) {
    J.sol = sol_s;
    if (J.local_trace && J.n_local_trace < J.local_trace_cap) {
      psulvsb_local_trace_t& T = J.local_trace[J.n_local_trace++];
      T.host_round = J.host_round;
      T.local_iter = J.local_iter_global;
      T.n_sampled_lines = (int)J.n_ls;
      T.n_sampled_points = J.n_sampled_pts;
      T.basic_choose = J.basic_choose;
      T.gnc_iterations = J.gnc_info[0];
      T.rot_inliers = J.gnc_info[1];
      T.n_rot_points = n_rot_pts;
      T.similar = similar;
      T.curr_count = curr_count;
      T.best_count = J.best_sampled_cnt;
      T.local_r = J.local_r;
      T.p_local = J.pro_local;
      T.l_rate = kLRate[J.rate_idx];
      T.b_rate = kBRate[J.rate_idx];
      T.scale = sol_s.s;
      for (int c = 0; c < 3; ++c)
        for (int r = 0; r < 3; ++r) T.R[c * 3 + r] = sol_s.R[r * 3 + c];
      for (int r = 0; r < 3; ++r) T.t[r] = sol_s.t[r];
    }
    J.local_iter_global += 1;
    base_s[0] = 0;
    base_s[1] = 0;
  }
  __syncthreads();

  if (J.pro_local > P.tpro_local && P.split_host_scoring) {
    // large M: engine_host_score_kernel (grid-wide) and engine_host_finish_kernel take over, in this tick
    if (tid == 0) {
      J.hs_curr = 0;
      J.phase = PHASE_HOST_SCORE;
    }
    return;
  }
  if (J.pro_local > P.tpro_local) {
    // ---- host scoring over all M correspondences + self-update decision (registration.cc:1399-1452)
    const Xform X = J.best_sampled;
    const uint32_t ev = (uint32_t)J.host_scorings;
    const int M = J.M;
    int curr = 0;
    // The two output lists (new correspondences, inlier map) are in ascending j.  The points go through in super-chunks
    // of 65 536: every warp leaves its decisions as two ballot words per 32 points in shared memory, then ONE block scan
    // per super-chunk places them (a scan per 1024 points was 98 scans and 200 barriers per host scoring at M = 100 000)
    constexpr int SUPER = 65536;
    __shared__ uint32_t addw_s[SUPER / 32], imapw_s[SUPER / 32];
    const int lane = tid & 31;
    for (int s0 = 0; s0 < M; s0 += SUPER) {
      const int s1 = min(M, s0 + SUPER);
      for (int j0 = s0; j0 < s1; j0 += BLK) {
        const int j = j0 + tid;
        int add = 0, imap = 0;
        if (j < s1) {
          int inl = 0;
          host_score_point(J, P, X, ev, j, add, imap, inl);
          curr += inl;
        }
        const unsigned int ab = __ballot_sync(0xffffffffu, add != 0), ib = __ballot_sync(0xffffffffu, imap != 0);
        if (lane == 0) {
          addw_s[(j0 - s0 + tid) >> 5] = ab;
          imapw_s[(j0 - s0 + tid) >> 5] = ib;
        }
      }
      __syncthreads();
      // thread t owns words 2t, 2t + 1 of the super-chunk (points s0 + 64 t .. + 63)
      const int nwords = (s1 - s0 + 31) >> 5;
      uint32_t wa[2], wi[2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int w = 2 * tid + k;
        // (the last word's bits past s1 are clear: add / imap are 0 for j >= s1; words past the chunk were not written)
        wa[k] = (w < nwords) ? addw_s[w] : 0u;
        wi[k] = (w < nwords) ? imapw_s[w] : 0u;
      }
      int ea, eb, ta, tb;
      block_scan2(&scratch, __popc(wa[0]) + __popc(wa[1]), __popc(wi[0]) + __popc(wi[1]), ea, eb, ta, tb);
      int pa = base_s[0] + ea, pi = base_s[1] + eb;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int jb = s0 + (2 * tid + k) * 32;
        for (uint32_t w = wa[k]; w; w &= w - 1) J.new_corr[pa++] = jb + __ffs(w) - 1;
        for (uint32_t w = wi[k]; w; w &= w - 1) J.inlier_map[pi++] = J.reduce_map[jb + __ffs(w) - 1];
      }
      __syncthreads();
      if (tid == 0) {
        base_s[0] += ta;
        base_s[1] += tb;
      }
      __syncthreads();
    }
    int dummy = 0;
    block_sum_int2(&scratch, curr, dummy);
    if (tid == 0) {
      finish_host_round(J, P, X, curr, elapsed_s, sb[blockIdx.x], gj[blockIdx.x], cq[blockIdx.x], n_done, base_s[0], base_s[1]);
    }
  } else if (tid == 0) {
    J.sampled_first_time = 0;
    if (J.local_iter_global >= P.max_local_iters) {
      J.status = PSULVSB_ERR_INTERNAL;  // non-terminating input (the reference would spin, registration.cc:903)
      J.phase = PHASE_DONE;
      sb[blockIdx.x].active = 0;
      gj[blockIdx.x].active = 0;
      cq[blockIdx.x].active = 0;
      atomicAdd(n_done, 1);
    } else {
      prepare_local(J, sb[blockIdx.x], gj[blockIdx.x], cq[blockIdx.x], P);
    }
  }
}

// ------------------------------------------------------------------------------------------
// split host scoring (large M): what the control kernel does in its last third, on the whole GPU.  One registration of
// 10^5 correspondences scored by ONE CTA -- a Philox draw and an erfc per outlier -- was ~ 0.3 ms of every tick.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLK)
    engine_host_score_kernel(JobCtl* __restrict__ jobs, EngineParams P) {
  JobCtl& J = jobs[blockIdx.y];
  if (J.phase != PHASE_HOST_SCORE) return;
  const int M = J.M;
  const int j0 = blockIdx.x * BLK;
  if (j0 >= M) return;
  const int j = j0 + threadIdx.x;
  const Xform X = J.best_sampled;
  const uint32_t ev = (uint32_t)J.host_scorings;
  int add = 0, imap = 0, inl = 0;
  if (j < M) host_score_point(J, P, X, ev, j, add, imap, inl);
  const unsigned int ab = __ballot_sync(0xffffffffu, add != 0), ib = __ballot_sync(0xffffffffu, imap != 0);
  const unsigned int nb = __ballot_sync(0xffffffffu, inl != 0);
  if ((threadIdx.x & 31) == 0 && j < M) {  // (a warp whose first point is past M has no word)
    const int nw = (M + 31) >> 5;
    J.hs_bits[j >> 5] = ab;
    J.hs_bits[nw + (j >> 5)] = ib;
    if (nb) atomicAdd(&J.hs_curr, __popc(nb));
  }
}

__global__ void __launch_bounds__(BLK)
    engine_host_finish_kernel(JobCtl* __restrict__ jobs, SampleJob* __restrict__ sb, GncJob* __restrict__ gj,
                              CliqueJob* __restrict__ cq, EngineParams P, double elapsed_s, int* __restrict__ n_done) {
  JobCtl& J = jobs[blockIdx.x];
  if (J.phase != PHASE_HOST_SCORE) return;
  __shared__ BlockScratch scratch;
  __shared__ int base_s[2];
  const int tid = threadIdx.x;
  const int M = J.M, nw = (M + 31) >> 5;
  if (tid == 0) base_s[0] = base_s[1] = 0;
  __syncthreads();
  // the two ordered lists from the decision bits: thread t owns words 2t, 2t + 1 of a super-chunk of 65 536 points
  constexpr int SUPER = 65536;
  for (int s0 = 0; s0 < M; s0 += SUPER) {
    uint32_t wa[2], wi[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int w = (s0 >> 5) + 2 * tid + k;
      wa[k] = (w < nw) ? J.hs_bits[w] : 0u;
      wi[k] = (w < nw) ? J.hs_bits[nw + w] : 0u;
    }
    int ea, eb, ta, tb;
    block_scan2(&scratch, __popc(wa[0]) + __popc(wa[1]), __popc(wi[0]) + __popc(wi[1]), ea, eb, ta, tb);
    int pa = base_s[0] + ea, pi = base_s[1] + eb;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int jb = s0 + (2 * tid + k) * 32;
      for (uint32_t w = wa[k]; w; w &= w - 1) J.new_corr[pa++] = jb + __ffs(w) - 1;
      for (uint32_t w = wi[k]; w; w &= w - 1) J.inlier_map[pi++] = J.reduce_map[jb + __ffs(w) - 1];
    }
    __syncthreads();
    if (tid == 0) {
      base_s[0] += ta;
      base_s[1] += tb;
    }
    __syncthreads();
  }
  if (tid == 0)
    finish_host_round(J, P, J.best_sampled, J.hs_curr, elapsed_s, sb[blockIdx.x], gj[blockIdx.x], cq[blockIdx.x], n_done,
                      base_s[0], base_s[1]);
}

// ------------------------------------------------------------------------------------------
// refinement (registration.cc:1499-1525: weightedSVD :526-569, calculateRMSE :571-602) + solution
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLK)
    engine_refine_kernel(JobCtl* __restrict__ jobs, psulvsb_solution_t* __restrict__ out,
                         const unsigned long long* __restrict__ border) {
  JobCtl& J = jobs[blockIdx.x];
  __shared__ BlockScratch scratch;
  __shared__ double Radj_s[9], tadj_s[3];
  const int tid = threadIdx.x;
  const int M = J.M;
  const Xform init = J.best_sampled;  // registration.cc:1508-1509 (best *sampled*, SURVEY defect 8)
  bool refined = false;
  Xform fin = J.best_host;
  if (J.valid && J.best_host_cnt != 0) {
    // T_init applied to the source, weighted centroids
    double acc[4] = {0, 0, 0, 0}, acc2[4] = {0, 0, 0, 0};
    for (int k = tid; k < M; k += BLK) {
      const double* p = J.ori_src + 3 * (size_t)k;
      const double* q = J.ori_dst + 3 * (size_t)k;
      const double w = (double)J.inlier_counter[k];
      acc[3] += w;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const double x = dadd(dadd(dadd(dmul(init.R[r * 3], p[0]), dmul(init.R[r * 3 + 1], p[1])), dmul(init.R[r * 3 + 2], p[2])), init.t[r]);
        acc[r] += x * w;
        acc2[r] += q[r] * w;
      }
    }
    block_sum<4>(&scratch, acc);
    block_sum<4>(&scratch, acc2);
    const double total = acc[3];
    double cs[3], ct[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      cs[r] = acc[r] / total;
      ct[r] = acc2[r] / total;
    }
    double cov[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) cov[i] = 0.0;
    for (int k = tid; k < M; k += BLK) {
      const double* p = J.ori_src + 3 * (size_t)k;
      const double* q = J.ori_dst + 3 * (size_t)k;
      const double w = (double)J.inlier_counter[k];
      if (w != 0.0) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const double x = dadd(dadd(dadd(dmul(init.R[r * 3], p[0]), dmul(init.R[r * 3 + 1], p[1])), dmul(init.R[r * 3 + 2], p[2])), init.t[r]);
          const double a = (x - cs[r]) * w;
#pragma unroll
          for (int c = 0; c < 3; ++c) cov[r * 3 + c] += a * (q[c] - ct[c]);
        }
      }
    }
    {
      double part[4];
      for (int g = 0; g < 3; ++g) {
        part[0] = cov[g * 3];
        part[1] = cov[g * 3 + 1];
        part[2] = cov[g * 3 + 2];
        part[3] = 0.0;
        block_sum<4>(&scratch, part);
        cov[g * 3] = part[0];
        cov[g * 3 + 1] = part[1];
        cov[g * 3 + 2] = part[2];
      }
    }
    if (tid == 0) {
      double H[3][3], Rf[3][3];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) H[r][c] = cov[r * 3 + c];
      kabsch_rotation(H, Rf);
      double tf[3];
      for (int r = 0; r < 3; ++r) tf[r] = ct[r] - ((Rf[r][0] * cs[0] + Rf[r][1] * cs[1]) + Rf[r][2] * cs[2]);
      // adj = [Rf tf] * [Rinit tinit]
      for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c)
          Radj_s[r * 3 + c] = (Rf[r][0] * init.R[0 * 3 + c] + Rf[r][1] * init.R[1 * 3 + c]) + Rf[r][2] * init.R[2 * 3 + c];
        tadj_s[r] = ((Rf[r][0] * init.t[0] + Rf[r][1] * init.t[1]) + Rf[r][2] * init.t[2]) + tf[r];
      }
    }
    __syncthreads();
    double e[4] = {0, 0, 0, 0};  // sse adj, sse ori, count
    for (int k = tid; k < M; k += BLK) {
      if (J.final_inliers[k] == 1) {
        const double* p = J.ori_src + 3 * (size_t)k;
        const double* q = J.ori_dst + 3 * (size_t)k;
        double sa = 0.0, so = 0.0;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const double xa = dadd(dadd(dadd(dmul(Radj_s[r * 3], p[0]), dmul(Radj_s[r * 3 + 1], p[1])), dmul(Radj_s[r * 3 + 2], p[2])), tadj_s[r]);
          const double xo = dadd(dadd(dadd(dmul(init.R[r * 3], p[0]), dmul(init.R[r * 3 + 1], p[1])), dmul(init.R[r * 3 + 2], p[2])), init.t[r]);
          const double da = xa - q[r], dor = xo - q[r];
          sa += da * da;
          so += dor * dor;
        }
        e[0] += sa;
        e[1] += so;
        e[2] += 1.0;
      }
    }
    block_sum<4>(&scratch, e);
    if (e[2] > 0.0) {
      const double adj_rmse = sqrt(e[0] / e[2]), ori_rmse = sqrt(e[1] / e[2]);
      refined = adj_rmse < ori_rmse;
    }
    if (refined) {
      for (int i = 0; i < 9; ++i) fin.R[i] = Radj_s[i];
      for (int r = 0; r < 3; ++r) fin.t[r] = tadj_s[r];
    }
  }
  if (tid == 0) {
    psulvsb_solution_t& S = out[blockIdx.x];
    S.valid = (J.valid && J.status == PSULVSB_OK) ? 1 : 0;
    S.scale = J.valid ? J.best_host.s : 1.0;
    S.final_inlier_count = J.valid ? J.best_host_cnt : 0;
    if (!J.valid) xform_identity(fin);
    if (J.aborted) {  // registration.cc:1032-1036: the solution fields keep the values of the last iteration
      fin = J.sol;
      S.scale = J.cur_scale;
    }
    for (int r = 0; r < 3; ++r) S.translation[r] = fin.t[r];
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) S.rotation[c * 3 + r] = fin.R[r * 3 + c];
    S.host_rounds = J.host_round;
    S.local_iters = J.local_iter_global;
    S.n_line_vectors = (long long)J.C0 * (J.C0 - 1) / 2;
    S.n_reduced = (long long)J.n_red0;
    S.final_C = J.C;
    S.refined = refined ? 1 : 0;
    S.escalations = J.escalations;
    S.borderline_pairs = border ? (long long)border[blockIdx.x] : 0;
    S.status = J.status;
    J.refined = refined ? 1 : 0;
  }
}

// copies of the per-point outputs a trace may ask for
__global__ void engine_export_points_kernel(const JobCtl* __restrict__ jobs, int job, int* __restrict__ final_inliers,
                                            int* __restrict__ inlier_counter) {
  const JobCtl& J = jobs[job];
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < J.M) {
    if (final_inliers) final_inliers[j] = J.final_inliers[j];
    if (inlier_counter) inlier_counter[j] = J.inlier_counter[j];
  }
}

}  // namespace psulvsb
