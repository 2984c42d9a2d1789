// Launch entry points.  The step kernels are spread over translation units so that the library builds in parallel: one
// per scenario (kern_step_<scenario>.cu) and one per scenario and compile-time team size (kern_team_<scenario><n>.cu).
#pragma once
#include "common.cuh"

namespace mrb {
// kern_team_<scenario><n>.cu exists for n = 8, 12, ..., team_kernel_max(scenario); 0 = none. The PredatorCapturePrey
// units also carry the QP-alone kernels of mrb_barrier_qp.
constexpr int team_kernel_max(int scn) { return scn == MRB_PCP ? 32 : scn == MRB_WAREHOUSE ? 12 : scn == MRB_SIMPLE ? 16 : 0; }
template <int SCN, int NC> cudaError_t launch_step_team(const Params &, const int32_t *, cudaStream_t, bool exact);
template <int NC> cudaError_t launch_qp_team(int N, int barrier_default, int64_t B, const double *, const double *, double *, int32_t *, cudaStream_t);

// the compile-time team size a team of N robots runs on: N rounded up to a multiple of four
constexpr int team_size(int N) { return (N + 3) & ~3; }
// launch(std::integral_constant<int, team_size(N)>()) if team_size(N) is one of 8, 12, ..., MAX
template <int MAX, int NC = 8, typename F>
cudaError_t with_team_size(int N, F &&launch)
{
    if constexpr (NC > MAX) return cudaErrorNotSupported;
    else return team_size(N) == NC ? launch(std::integral_constant<int, NC>()) : with_team_size<MAX, NC + 4>(N, launch);
}

template <int SCN> cudaError_t launch_step(const Params &p, const int32_t *actions, cudaStream_t s);   // kern_step_<scenario>.cu
cudaError_t launch_reset(const Params &p, const uint8_t *mask, cudaStream_t s);
cudaError_t launch_barrier_qp(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u,
                              int32_t *iters, cudaStream_t s);
// explore.cu: the selection kernel, then a one-thread kernel that advances *step
cudaError_t launch_select_actions(int64_t num_envs, int32_t n_agents, int32_t n_actions, const mrb_select_desc &desc,
                                  int64_t *step, const float *q, int32_t *actions, cudaStream_t s);
// record.cu: mrb_record_begin (begin, actions unused) and mrb_record_step, one launch each
cudaError_t launch_record(const Params &p, int n_actions, const mrb_episode_batch &batch, bool begin,
                          const int32_t *actions, cudaStream_t s);
// compact.cu: mrb_step_masked's list of active envs.  work i32 [3]: count (out), then two words that must be 0 on entry
// and are 0 again on exit
cudaError_t launch_compact(const uint8_t *active, int64_t B, int32_t *envs, int32_t *work, cudaStream_t s);
// eval.cu: mrb_eval_begin (begin) and mrb_eval_step, one launch each
cudaError_t launch_eval(const Params &p, const mrb_eval_table &table, bool begin, cudaStream_t s);
}  // namespace mrb
