// Exploratory action selection over the policy's output (mrb_select_actions): EPyMARL's EpsilonGreedyActionSelector
// with its linear DecayThenFlatSchedule, and SoftPoliciesSelector's draw from softmax(q).  Kept apart from the policy
// kernels so that their greedy results and register budgets do not change.
//
// Random numbers: one Philox4x32-10 block per (env, agent, step), key = seed, counter = (global env id lo, hi,
// (uint32) t, 0x80000000 | agent).  The reset streams use counter (env id, episode, block) with a small block word, so
// the top bit keeps the two families apart.  The global env id makes every draw independent of how the envs are
// sharded over devices; t is the 64-bit device counter, so the counter word wraps after 2^32 steps.
#include "launchers.h"

namespace mrb {

__global__ void __launch_bounds__(256)
select_actions_kernel(int64_t rows, int32_t n_agents, int32_t n_actions, int32_t mode, uint64_t seed, int64_t env_id0,
                      double eps_start, double eps_finish, int64_t anneal_time, const int64_t *__restrict__ step,
                      const float *__restrict__ q, int32_t *__restrict__ actions)
{
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    const int64_t t = *step;
    const int64_t env = row / n_agents;
    const uint32_t agent = (uint32_t)(row - env * n_agents);
    Philox rng(seed, (uint64_t)(env_id0 + env), (uint32_t)t);
    rng.c3 = 0x80000000u | agent;
    rng.refill();
    const uint32_t w0 = rng.buf[0], w1 = rng.buf[1], w2 = rng.buf[2], w3 = rng.buf[3];

    if (mode == MRB_SELECT_EPSILON_GREEDY) {
        const double eps = fmax(eps_finish, eps_start - (eps_start - eps_finish) * (double)t / (double)anneal_time);
        const uint64_t thr = eps >= 1.0 ? (1ull << 32) : (uint64_t)floor(eps * 4294967296.0);
        if (w0 < thr) actions[row] = (int32_t)(((uint64_t)w1 * (uint32_t)n_actions) >> 32);
        return;
    }
    // softmax: the first action whose running sum of exp(q - max q) exceeds u * S, all in double
    const float *qr = q + row * n_actions;
    float m = qr[0];
    for (int a = 1; a < n_actions; a++) m = fmaxf(m, qr[a]);
    double S = 0.0;
    for (int a = 0; a < n_actions; a++) S += exp((double)qr[a] - (double)m);
    const double target = (((double)(w2 >> 5) * 67108864.0 + (double)(w3 >> 6)) / 9007199254740992.0) * S;
    double c = 0.0;
    int pick = -1, last = 0;
    for (int a = 0; a < n_actions; a++) {
        const double e = exp((double)qr[a] - (double)m);
        c += e;
        if (e > 0.0) last = a;
        if (pick < 0 && c > target) pick = a;
    }
    actions[row] = pick >= 0 ? pick : last;       // rounding can leave c <= target after the last action
}

__global__ void advance_step_kernel(int64_t *step) { *step += 1; }

cudaError_t launch_select_actions(int64_t num_envs, int32_t n_agents, int32_t n_actions, const mrb_select_desc &d,
                                  int64_t *step, const float *q, int32_t *actions, cudaStream_t s)
{
    const int tpb = 256;
    const int64_t rows = num_envs * n_agents;
    select_actions_kernel<<<(unsigned)((rows + tpb - 1) / tpb), tpb, 0, s>>>(
        rows, n_agents, n_actions, d.mode, d.seed, d.env_id0, d.eps_start, d.eps_finish, d.anneal_time, step, q, actions);
    cudaError_t st = cudaGetLastError();
    if (st != cudaSuccess) return st;
    advance_step_kernel<<<1, 1, 0, s>>>(step);
    return cudaGetLastError();
}

}  // namespace mrb
