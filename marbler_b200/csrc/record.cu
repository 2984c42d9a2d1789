// Episode recording (mrb_record_begin / mrb_record_step): the writes EPyMARL's ParallelRunner makes into its
// EpisodeBatch, one launch per env step.  Pure data movement, kept out of the step kernels so that their register
// budgets and results do not change.
//
// A CTA takes kEnvs consecutive envs.  One thread per env reads and advances that env's cursor and writes its
// per-env scalars (reward, terminated, filled); then the whole CTA writes the rows, consecutive threads on consecutive
// elements: the obs rows of the tile are E*N*D contiguous floats in, and each env's row is N*W contiguous floats out,
// so every warp access is coalesced.  Every access is scalar at the element's own width (the alignment
// mrb_record_begin / mrb_record_step check).
#include "launchers.h"

namespace mrb {

static constexpr int kThreads = 256, kEnvs = 32;

// f(e, a, c) for every element (env e < E, sub-row a < n, column c < S) of a tile, element (e*n + a)*S + c on thread
// (element mod kThreads).  The indices advance by kThreads elements per iteration without a division.
template <typename F>
__device__ __forceinline__ void for_tile(int E, int n, int S, F &&f)
{
    const int row = n * S, total = E * row;
    int i = threadIdx.x;
    if (i >= total) return;
    int e = i / row, k = i - e * row, a = k / S, c = k - a * S;
    const int de = kThreads / row, dk = kThreads - de * row, da = dk / S, dc = dk - da * S;
    for (; i < total; i += kThreads) {
        f(e, a, c);
        c += dc, a += da, e += de;
        if (c >= S) c -= S, a++;
        if (a >= n) a -= n, e++;
    }
}

// Per env, the call writes row `ra` of actions / actions_onehot / reward / terminated and row `ro` of obs /
// avail_actions / filled (-1: nothing).  `src`: the values come from the env's buffers (an active env's step);
// otherwise they are zero.  `open`: avail_actions and filled of row `ro` are 1 (row 0, or a step of an active env).
__global__ void __launch_bounds__(kThreads)
record_kernel(mrb_episode_batch b, int64_t B, int N, int D, int A, int W, int T, bool begin,
              const float *__restrict__ obs, const float *__restrict__ reward, const uint8_t *__restrict__ done,
              const int32_t *__restrict__ actions)
{
    __shared__ int s_ra[kEnvs], s_ro[kEnvs];
    __shared__ bool s_src[kEnvs], s_open[kEnvs];
    const int64_t env0 = (int64_t)blockIdx.x * kEnvs, R = (int64_t)T + 1;
    const int E = B - env0 < kEnvs ? (int)(B - env0) : kEnvs;
    if ((int)threadIdx.x < E) {
        const int e = threadIdx.x;
        const int64_t env = env0 + e;
        if (begin) {
            s_ra[e] = T, s_ro[e] = 0, s_src[e] = false, s_open[e] = true;
            b.reward[env * R + T] = 0.0f;
            b.terminated[env * R + T] = 0;
            b.filled[env * R] = 1;
            b.cursor[env] = 0;
        } else {
            const int32_t cur = b.cursor[env];
            const bool active = cur >= 0;
            const int t = active ? cur : ~cur;
            s_ra[e] = t < T ? t : -1, s_ro[e] = t < T ? t + 1 : -1, s_src[e] = active, s_open[e] = active;
            if (t < T) {
                float r = 0.0f;
                bool term = false;
                if (active) {
                    const float *rw = reward + env * N;
                    r = rw[0];
                    for (int a = 1; a < N; a++) r = __fadd_rn(r, rw[a]);       // agent index order, no reassociation
                    term = done[env] != 0 || t + 1 >= T;
                }
                b.reward[env * R + t] = r;
                b.terminated[env * R + t] = term;
                b.filled[env * R + t + 1] = active;
                b.cursor[env] = active && !term ? t + 1 : ~(t + 1);
            }
        }
    }
    __syncthreads();

    const int NW = N * W, NA = N * A;
    const float *obs_tile = obs + env0 * N * D;
    const int32_t *act_tile = actions + env0 * N;
    for_tile(E, N, W, [&](int e, int a, int c) {
        const int ro = s_ro[e];
        if (ro < 0) return;
        const float v = s_src[e] && c < D ? obs_tile[(e * N + a) * D + c] : 0.0f;
        b.obs[((env0 + e) * R + ro) * NW + a * W + c] = v;
    });
    for_tile(E, N, 1, [&](int e, int a, int) {
        const int ra = s_ra[e];
        if (ra < 0) return;
        b.actions[((env0 + e) * R + ra) * N + a] = s_src[e] ? act_tile[e * N + a] : 0;
    });
    for_tile(E, N, A, [&](int e, int a, int c) {
        const int ra = s_ra[e], ro = s_ro[e];
        if (ra >= 0) b.actions_onehot[((env0 + e) * R + ra) * NA + a * A + c] = s_src[e] && act_tile[e * N + a] == c ? 1.0f : 0.0f;
        if (ro >= 0) b.avail_actions[((env0 + e) * R + ro) * NA + a * A + c] = s_open[e];
    });
}

cudaError_t launch_record(const Params &p, int n_actions, const mrb_episode_batch &b, bool begin,
                          const int32_t *actions, cudaStream_t s)
{
    const int64_t B = p.B;
    record_kernel<<<(unsigned)((B + kEnvs - 1) / kEnvs), kThreads, 0, s>>>(
        b, B, p.cfg.num_robots, p.obs_dim, n_actions, b.obs_width, b.episode_limit, begin, p.buf.obs, p.buf.reward,
        p.buf.done, actions);
    return cudaGetLastError();
}

}  // namespace mrb
