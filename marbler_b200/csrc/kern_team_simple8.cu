#include "kern_team.cuh"
namespace mrb {
template cudaError_t launch_step_team<MRB_SIMPLE, 8>(const Params &, const int32_t *, cudaStream_t, bool);
}  // namespace mrb
