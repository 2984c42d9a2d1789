// Evaluation (mrb_eval_begin / mrb_eval_step): each env's first K finished episodes into a per-episode results
// table, one launch per env step.  Kept out of the step kernels so that their register budgets and results do not
// change; it reads only the output buffers the step kernel has just written (auto-reset leaves them alone).
//
// One thread per env.  The per-env scalars (done, message, remaining, the accumulators, count) are coalesced; the
// N rewards and dists of an env are contiguous, so a warp's loads of them cover 32 * N consecutive floats.
#include "launchers.h"

namespace mrb {

static constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads)
eval_kernel(mrb_eval_table t, int64_t B, int N, int max_steps, bool begin, const float *__restrict__ reward,
            const uint8_t *__restrict__ done, const uint8_t *__restrict__ message,
            const int32_t *__restrict__ remaining, const float *__restrict__ dist)
{
    const int64_t env = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (env >= B) return;
    if (begin) {
        t.acc_return[env] = 0.0;
        t.acc_length[env] = 0;
        t.acc_dist[env] = 0.0;
        t.count[env] = 0;
        return;
    }
    const float *rw = reward + env * N;
    float team = 0.f;
    for (int a = 0; a < N; a++) team = __fadd_rn(team, rw[a]);     // agent index order, as the step kernel's return
    double d = 0.0;
    if (dist) {
        const float *dw = dist + env * N;
        for (int a = 0; a < N; a++) d = __dadd_rn(d, (double)dw[a]);
    }
    const double ret = __dadd_rn(t.acc_return[env], (double)team), dd = __dadd_rn(t.acc_dist[env], d);
    const int32_t len = t.acc_length[env] + 1;
    if (!done[env]) {
        t.acc_return[env] = ret;
        t.acc_length[env] = len;
        t.acc_dist[env] = dd;
        return;
    }
    const int32_t k = t.count[env];
    if (k < t.episodes) {
        const int64_t row = env * t.episodes + k;
        const uint8_t msg = message[env];
        t.return_[row] = ret;
        t.length[row] = len;
        t.message[row] = msg;
        t.timeout[row] = msg == 0 && len > max_steps;
        t.remaining[row] = remaining[env];
        t.dist[row] = (float)dd;
        t.count[env] = k + 1;
    }
    t.acc_return[env] = 0.0;
    t.acc_length[env] = 0;
    t.acc_dist[env] = 0.0;
}

cudaError_t launch_eval(const Params &p, const mrb_eval_table &t, bool begin, cudaStream_t s)
{
    const int64_t B = p.B;
    eval_kernel<<<(unsigned)((B + kThreads - 1) / kThreads), kThreads, 0, s>>>(
        t, B, p.cfg.num_robots, p.cfg.max_episode_steps, begin, p.buf.reward, p.buf.done, p.buf.message,
        p.buf.remaining, p.buf.dist);
    return cudaGetLastError();
}

}  // namespace mrb
