// engine_kernels.cuh -- control kernels of the lock-step batch engine (engine_kernels.cu).
#pragma once

#include "engine.cuh"
#include "engine_state.cuh"

namespace psulvsb {

constexpr int kCtlThreads = 1024;  // block size of every control kernel (== BLK in solve_dev.cuh)

__global__ void engine_init_kernel(JobCtl* jobs, SampleJob* sl, SampleJob* sb, GncJob* gj, CliqueJob* cq,
                                   const unsigned long long* n_edges, EngineParams P, int* n_done);
// the round-start kernel over n_jobs registrations; narrow: JobCtl::edges are EdgeNarrow lists, else EdgeWide
int launch_round_start(cudaStream_t st, int n_jobs, JobCtl* jobs, SampleJob* sl, SampleJob* sb, GncJob* gj, CliqueJob* cq,
                       const EngineParams& P, int* n_done, bool narrow);
__global__ void engine_scale_kernel(JobCtl* jobs, GncJob* gj, CliqueJob* cq, EngineParams P);
__global__ void engine_local_control_kernel(JobCtl* jobs, SampleJob* sl, SampleJob* sb, GncJob* gj, CliqueJob* cq,
                                            EngineParams P, double elapsed_s, int* n_done);
__global__ void engine_host_score_kernel(JobCtl* jobs, EngineParams P);
__global__ void engine_host_finish_kernel(JobCtl* jobs, SampleJob* sb, GncJob* gj, CliqueJob* cq, EngineParams P,
                                          double elapsed_s, int* n_done);
__global__ void engine_refine_kernel(JobCtl* jobs, psulvsb_solution_t* out, const unsigned long long* border);
__global__ void engine_export_points_kernel(const JobCtl* jobs, int job, int* final_inliers, int* inlier_counter);

}  // namespace psulvsb
