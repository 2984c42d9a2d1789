// Shared body of the per-scenario launch translation units (kern_step_*.cu).
#pragma once
#include "launchers.h"
#include "step_thread.cuh"
#include "step_warp.cuh"

namespace mrb {

template <int SCN, int N>
inline cudaError_t launch_thread(const Params &p, const int32_t *actions, cudaStream_t s)
{
    constexpr int tpb = ThreadShape<N>::kThreads;
    const unsigned grid = (unsigned)((p.env_hi - p.env_lo + tpb - 1) / tpb);
    constexpr size_t smem = QpStore<N>::kBytes;
    if (smem > 48 * 1024) {
        const cudaError_t attr = cudaFuncSetAttribute(step_thread_kernel<SCN, N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (attr != cudaSuccess) return attr;
    }
    step_thread_kernel<SCN, N><<<grid, tpb, smem, s>>>(p, actions);
    return cudaGetLastError();
}

// teams of 2..6 robots: one env per thread; anything else up to 32 robots: one env per warp
template <int SCN>
inline cudaError_t launch_step_generic(const Params &p, const int32_t *actions, cudaStream_t s, bool *launched)
{
    *launched = true;
    switch (p.cfg.num_robots) {
    case 2: if (SCN != MRB_MATERIAL) return launch_thread<SCN, (SCN != MRB_MATERIAL ? 2 : 4)>(p, actions, s); break;
    case 3: if (SCN != MRB_MATERIAL) return launch_thread<SCN, (SCN != MRB_MATERIAL ? 3 : 4)>(p, actions, s); break;
    case 4: return launch_thread<SCN, 4>(p, actions, s);
    case 5: return launch_thread<SCN, 5>(p, actions, s);
    case 6: return launch_thread<SCN, 6>(p, actions, s);
    default: break;
    }
    if (SCN == MRB_ARCTIC) { *launched = false; return cudaSuccess; }
    return launch_step_warp<SCN>(p, actions, s);
}

}  // namespace mrb
