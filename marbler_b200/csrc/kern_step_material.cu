#include "step_warp.cuh"
namespace mrb {
template cudaError_t launch_step<MRB_MATERIAL>(const Params &, const int32_t *, cudaStream_t);
}  // namespace mrb
