// Dispatch to the kernels with a compile-time size of the Newton system (kern_team_*.cu: FP64 tensor-core solver).  A
// team of N robots runs on the size rounded up to a multiple of four -- folded into the code when N is that multiple,
// padded with phantom robots otherwise -- if the scenario has a kernel of that size; every other case (and
// MRB_WARP_GENERIC=1) runs the run-time team size kernels of step_warp.cuh.  Measured (PredatorCapturePrey, ms per
// step of 32,768 envs, run-time vs compile-time size): 8 robots 5.81 vs 3.34, 12: 10.6 vs 5.81, 16: 15.1 vs 9.09,
// 20: 29.0 vs 13.7; 16,384 envs: 24 robots 31.6 vs 12.5, 28: 56.6 vs 16.5; padded: 10 robots (on 12) 3.90 vs 2.97,
// 18 (on 20) 12.6 vs 7.2, 23 (on 24) 22.3 vs 13.4; 20 robots padded variant 14.5 vs 13.7 folded.
// Kernels exist for PredatorCapturePrey 8..32, Warehouse 8 and 12, Simple 8..16 (what their spawn grids hold).
#include "launchers.h"

namespace mrb {
cudaError_t launch_step_team_pcp_8(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_pcp_12(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_pcp_16(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_pcp_20(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_pcp_24(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_pcp_28(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_pcp_32(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_warehouse_8(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_warehouse_12(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_simple_8(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_simple_12(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_step_team_simple_16(const Params &p, const int32_t *actions, cudaStream_t s, bool exact);
cudaError_t launch_qp_team_n_8(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);
cudaError_t launch_qp_team_n_12(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);
cudaError_t launch_qp_team_n_16(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);
cudaError_t launch_qp_team_n_20(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);
cudaError_t launch_qp_team_n_24(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);
cudaError_t launch_qp_team_n_28(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);
cudaError_t launch_qp_team_n_32(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s);

cudaError_t launch_step_team(int scenario, const Params &p, const int32_t *actions, cudaStream_t s, bool *handled)
{
    const int N = p.cfg.num_robots, size = (N + 3) & ~3;
    const bool exact = size == N;
    *handled = true;
    if (scenario == MRB_PCP) switch (size) {
    case 8: return launch_step_team_pcp_8(p, actions, s, exact);
    case 12: return launch_step_team_pcp_12(p, actions, s, exact);
    case 16: return launch_step_team_pcp_16(p, actions, s, exact);
    case 20: return launch_step_team_pcp_20(p, actions, s, exact);
    case 24: return launch_step_team_pcp_24(p, actions, s, exact);
    case 28: return launch_step_team_pcp_28(p, actions, s, exact);
    case 32: return launch_step_team_pcp_32(p, actions, s, exact);
    default: break;
    }
    if (scenario == MRB_WAREHOUSE) switch (size) {
    case 8: return launch_step_team_warehouse_8(p, actions, s, exact);
    case 12: return launch_step_team_warehouse_12(p, actions, s, exact);
    default: break;
    }
    if (scenario == MRB_SIMPLE) switch (size) {
    case 8: return launch_step_team_simple_8(p, actions, s, exact);
    case 12: return launch_step_team_simple_12(p, actions, s, exact);
    case 16: return launch_step_team_simple_16(p, actions, s, exact);
    default: break;
    }
    *handled = false;
    return cudaSuccess;
}

cudaError_t launch_qp_team(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters,
                           cudaStream_t s, bool *handled)
{
    *handled = true;
    switch ((N + 3) & ~3) {
    case 8: return launch_qp_team_n_8(N, barrier_default, B, dxi, xi, u, iters, s);
    case 12: return launch_qp_team_n_12(N, barrier_default, B, dxi, xi, u, iters, s);
    case 16: return launch_qp_team_n_16(N, barrier_default, B, dxi, xi, u, iters, s);
    case 20: return launch_qp_team_n_20(N, barrier_default, B, dxi, xi, u, iters, s);
    case 24: return launch_qp_team_n_24(N, barrier_default, B, dxi, xi, u, iters, s);
    case 28: return launch_qp_team_n_28(N, barrier_default, B, dxi, xi, u, iters, s);
    case 32: return launch_qp_team_n_32(N, barrier_default, B, dxi, xi, u, iters, s);
    default: break;
    }
    *handled = false;
    return cudaSuccess;
}
}  // namespace mrb
