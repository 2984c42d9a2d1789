// Bodies of launch_step_team and launch_qp_team (launchers.h), explicitly instantiated in kern_team_<scenario><n>.cu: one
// translation unit per (scenario, compile-time size of the Newton system) holds the warp kernel with the FP64 tensor-core
// solver (QpWarp<PPL, NC, EXACT>::factor_tiles / solve_tiles) in two variants -- exactly NC robots (team size folded into
// the code) and N <= NC robots at run time (phantom robots pad the last tile).  The PredatorCapturePrey unit of a size
// also carries the QP-alone kernels (mrb_barrier_qp).
#pragma once
#include "step_warp.cuh"

namespace mrb {
template <int SCN, int NC>
cudaError_t launch_step_team(const Params &p, const int32_t *actions, cudaStream_t s, bool exact)
{
    if (exact) return launch_step_warp_ppl<SCN, team_ppl(NC), NC, true>(p, actions, s);
    return launch_step_warp_ppl<SCN, team_ppl(NC), NC, false>(p, actions, s);
}

template <int NC>
cudaError_t launch_qp_team(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u,
                           int32_t *iters, cudaStream_t s)
{
    if (N == NC) return launch_qp_warp_ppl<team_ppl(NC), NC, true>(N, barrier_default, B, dxi, xi, u, iters, s);
    return launch_qp_warp_ppl<team_ppl(NC), NC, false>(N, barrier_default, B, dxi, xi, u, iters, s);
}
}  // namespace mrb
