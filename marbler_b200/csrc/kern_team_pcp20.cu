#include "kern_team.cuh"
namespace mrb {
template cudaError_t launch_step_team<MRB_PCP, 20>(const Params &, const int32_t *, cudaStream_t, bool);
template cudaError_t launch_qp_team<20>(int, int, int64_t, const double *, const double *, double *, int32_t *, cudaStream_t);
}  // namespace mrb
