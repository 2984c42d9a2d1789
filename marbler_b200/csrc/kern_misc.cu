// reset kernels and the stand-alone barrier-QP kernels
#include "launchers.h"
#include "step_thread.cuh"
#include "step_warp.cuh"

namespace mrb {

template <int SCN>
static cudaError_t launch_reset_scn(const Params &p, const uint8_t *mask, cudaStream_t s)
{
    const int tpb = 128;
    reset_kernel<SCN><<<(unsigned)((p.env_hi - p.env_lo + tpb - 1) / tpb), tpb, 0, s>>>(p, mask);
    return cudaGetLastError();
}

cudaError_t launch_reset(const Params &p, const uint8_t *mask, cudaStream_t s)
{
    switch (p.cfg.scenario) {
    case MRB_PCP: return launch_reset_scn<MRB_PCP>(p, mask, s);
    case MRB_WAREHOUSE: return launch_reset_scn<MRB_WAREHOUSE>(p, mask, s);
    case MRB_MATERIAL: return launch_reset_scn<MRB_MATERIAL>(p, mask, s);
    case MRB_ARCTIC: return launch_reset_scn<MRB_ARCTIC>(p, mask, s);
    default: return launch_reset_scn<MRB_SIMPLE>(p, mask, s);
    }
}

template <int N>
__global__ void __launch_bounds__(ThreadShape<N>::kThreads)
qp_thread_kernel(int64_t B, int barrier_default, const double *__restrict__ dxi, const double *__restrict__ xi,
                 double *__restrict__ u, int32_t *__restrict__ iters)
{
    const int64_t e = (int64_t)blockIdx.x * ThreadShape<N>::kThreads + threadIdx.x;
    if (e >= B) return;
    double xix[N], xiy[N], ux[N], uy[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
        xix[i] = xi[i * B + e]; xiy[i] = xi[(N + i) * B + e];
        ux[i] = dxi[i * B + e]; uy[i] = dxi[(N + i) * B + e];
    }
    const int it = qp_run<N>(xix, xiy, ux, uy, barrier_default != 0, QpStore<N>());
#pragma unroll
    for (int i = 0; i < N; i++) { u[i * B + e] = ux[i]; u[(N + i) * B + e] = uy[i]; }
    if (iters) iters[e] = it;
}

template <int N>
static cudaError_t launch_qp_thread(int64_t B, int barrier_default, const double *dxi, const double *xi,
                                    double *u, int32_t *iters, cudaStream_t s)
{
    constexpr size_t smem = QpStore<N>::kBytes;
    constexpr int tpb = ThreadShape<N>::kThreads;
    const unsigned grid = (unsigned)((B + tpb - 1) / tpb);
    if (smem > 48 * 1024) {
        const cudaError_t attr = cudaFuncSetAttribute(qp_thread_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (attr != cudaSuccess) return attr;
    }
    qp_thread_kernel<N><<<grid, tpb, smem, s>>>(B, barrier_default, dxi, xi, u, iters);
    return cudaGetLastError();
}

cudaError_t launch_barrier_qp(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u,
                              int32_t *iters, cudaStream_t s)
{
    switch (N) {
    case 2: return launch_qp_thread<2>(B, barrier_default, dxi, xi, u, iters, s);
    case 3: return launch_qp_thread<3>(B, barrier_default, dxi, xi, u, iters, s);
    case 4: return launch_qp_thread<4>(B, barrier_default, dxi, xi, u, iters, s);
    case 5: return launch_qp_thread<5>(B, barrier_default, dxi, xi, u, iters, s);
    case 6: return launch_qp_thread<6>(B, barrier_default, dxi, xi, u, iters, s);
    default: break;
    }
    // one robot (no pair constraint) and MRB_WARP_GENERIC: the run-time team size kernel; 7..32 robots: the tensor-core
    // kernels of the PredatorCapturePrey team units
    if (N >= 7 && team_size(N) <= team_kernel_max(MRB_PCP) && !warp_generic())
        return with_team_size<team_kernel_max(MRB_PCP)>(N, [&](auto nc) { return launch_qp_team<nc>(N, barrier_default, B, dxi, xi, u, iters, s); });
    return with_runtime_ppl(N, [&](auto ppl) { return launch_qp_warp_ppl<ppl>(N, barrier_default, B, dxi, xi, u, iters, s); });
}

}  // namespace mrb
