// Stream compaction of mrb_step_masked: the active mask u8 [B] -> the ids of the active envs (ascending within each
// CTA's slice; the slices land in the order the CTAs reach the running total) and their number.  The step kernels then
// run one item per listed env, so the live envs fill whole warps however the finished ones are scattered.
//
// One launch, no memset: each CTA reserves its slice of the list with one atomicAdd on a running total, and the last CTA
// to finish (a ticket counter) publishes the total as the count and puts the total and the ticket back to 0 for the
// next launch.
#include "launchers.h"

namespace mrb {

static constexpr int kThreads = 256, kWarps = kThreads / 32;

// work: [0] count (out), [1] running total, [2] CTAs finished; [1] and [2] are 0 between launches
__global__ void __launch_bounds__(kThreads)
compact_kernel(const uint8_t *__restrict__ active, int64_t B, int32_t *__restrict__ envs, int32_t *__restrict__ work)
{
    __shared__ int warp_off[kWarps], base;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const bool a = e < B && active[e] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, a);
    if (lane == 0) warp_off[w] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
        for (int k = 0; k < kWarps; k++) { const int n = warp_off[k]; warp_off[k] = total; total += n; }
        base = total ? atomicAdd(work + 1, total) : 0;
        __threadfence();                            // this CTA's share of the total is in before its ticket
        if (atomicAdd(work + 2, 1) == (int)gridDim.x - 1) {
            work[0] = atomicExch(work + 1, 0);
            work[2] = 0;
        }
    }
    __syncthreads();
    if (a) envs[base + warp_off[w] + __popc(m & ((1u << lane) - 1u))] = (int32_t)e;
}

cudaError_t launch_compact(const uint8_t *active, int64_t B, int32_t *envs, int32_t *work, cudaStream_t s)
{
    compact_kernel<<<(unsigned)((B + kThreads - 1) / kThreads), kThreads, 0, s>>>(active, B, envs, work);
    return cudaGetLastError();
}

}  // namespace mrb
