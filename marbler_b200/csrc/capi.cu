// C ABI of libmarbler_b200.so (see include/marbler_b200.h).  Host side only validates, fills the
// kernel parameter block and launches; all arithmetic is in the kernels.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

#include "common.cuh"
#include "handle.h"
#include "launchers.h"

using namespace mrb;

static std::string g_create_error;
static std::atomic<int64_t> g_launches{0};
namespace mrb {
void count_launch() { g_launches++; }
int fail(mrb_env *e, int code, const std::string &msg)
{
    if (e) e->err = msg; else g_create_error = msg;
    return code;
}
int cuda_fail(mrb_env *e, cudaError_t st, const char *what)
{
    return fail(e, MRB_E_CUDA, std::string(what) + ": " + cudaGetErrorString(st));
}
}  // namespace mrb

// largest t with fl(sqrt(t)) <= r: sqrt(d2) <= r  <=>  d2 <= t for every double d2 >= 0
static double thr2(double r)
{
    if (!(r > 0.0)) return 0.0;
    double t = r * r;
    while (std::sqrt(t) > r) t = std::nextafter(t, 0.0);
    while (std::sqrt(std::nextafter(t, INFINITY)) <= r) t = std::nextafter(t, INFINITY);
    return t;
}

static int obs_block_count(const mrb_config &c)
{
    const int others = c.num_robots - 1;
    return 1 + (c.num_neighbors >= others ? others : c.num_neighbors);
}
static int obs_dim_of(const mrb_config &c)
{
    switch (c.scenario) {
    case MRB_PCP: return (c.capability_aware ? 6 : 4) * obs_block_count(c);       // PredatorCapturePrey.py:30-33,52
    case MRB_WAREHOUSE: return 3 * obs_block_count(c);                             // warehouse.py:52,70
    case MRB_MATERIAL: return c.capability_aware ? 11 : 9;                         // MaterialTransport.py:55-58
    case MRB_ARCTIC: return 30;                                                    // ArcticTransport.py:19
    default: return 2 * (c.num_robots + 1);                                        // simple.py:98
    }
}

extern "C" int mrb_version(void) { return MRB_ABI_VERSION; }
extern "C" int64_t mrb_launch_count(void) { return g_launches.load(); }

extern "C" const char *mrb_last_error(const mrb_env *env) { return env ? env->err.c_str() : g_create_error.c_str(); }

extern "C" int mrb_create(const mrb_config *cfg, int device, int64_t num_envs, int64_t env_id0, mrb_env **out)
{
    if (!cfg || !out) return fail(nullptr, MRB_E_ARG, "mrb_create: null argument");
    if (cfg->struct_size != (int32_t)sizeof(mrb_config))
        return fail(nullptr, MRB_E_ARG, "mrb_create: mrb_config.struct_size does not match this library (ABI mismatch)");
    const mrb_config &c = *cfg;
    if (c.scenario < MRB_PCP || c.scenario > MRB_SIMPLE) return fail(nullptr, MRB_E_ARG, "mrb_create: unknown scenario");
    // one robot has no pair constraint: rps' certificate would hand cvxopt an empty G, which the reference never does
    if (c.num_robots < 2 || c.num_robots > MRB_MAX_ROBOTS) return fail(nullptr, MRB_E_ARG, "mrb_create: num_robots must be in [2, 32]");
    if (!(c.collision_diameter > 0.0) || !(c.collision_offset >= 0.0) || !std::isfinite(c.collision_diameter + c.collision_offset))
        return fail(nullptr, MRB_E_ARG, "mrb_create: collision_diameter must be > 0 and collision_offset >= 0 (rps: 0.135 and 0 or 0.025)");
    if (num_envs < 1 || num_envs > INT32_MAX) return fail(nullptr, MRB_E_ARG, "mrb_create: num_envs must be in [1, 2^31)");
    if (c.update_frequency < 1 || c.ctrl_period < 1) return fail(nullptr, MRB_E_ARG, "mrb_create: update_frequency / ctrl_period must be >= 1");
    if (c.scenario == MRB_PCP && (c.num_prey < 1 || c.num_prey > MRB_MAX_PREY || c.num_predators < 0 || c.num_predators > c.num_robots))
        return fail(nullptr, MRB_E_ARG, "mrb_create: PredatorCapturePrey needs 1..32 prey and predators <= robots");
    if (c.scenario == MRB_ARCTIC && c.num_robots != 4)
        return fail(nullptr, MRB_E_ARG, "mrb_create: ArcticTransport is defined for exactly 4 robots (ArcticTransport.py:25-33)");
    if (c.scenario == MRB_MATERIAL && c.num_robots < 4)
        return fail(nullptr, MRB_E_ARG, "mrb_create: MaterialTransport reads 4 messages (MaterialTransport.py:119-120)");
    if ((c.scenario == MRB_PCP || c.scenario == MRB_WAREHOUSE) && c.num_neighbors < 0)
        return fail(nullptr, MRB_E_ARG, "mrb_create: num_neighbors must be >= 0");
    if (c.scenario != MRB_ARCTIC) {
        const mrb_spawn &s = c.spawn_robots;
        if (s.count != c.num_robots || s.xr * s.yr <= s.count || s.xr * s.yr > 64)
            return fail(nullptr, MRB_E_ARG, "mrb_create: robot spawn grid must have more cells than robots (rps assert) and at most 64");
    }
    if (c.scenario == MRB_PCP || c.scenario == MRB_SIMPLE) {
        const mrb_spawn &s = c.spawn_other;
        const int want = c.scenario == MRB_PCP ? c.num_prey : 1;
        if (s.count != want || s.xr * s.yr <= s.count || s.xr * s.yr > 64)
            return fail(nullptr, MRB_E_ARG, "mrb_create: prey/goal spawn grid must have more cells than items and at most 64");
    }
    int ndev = 0;
    cudaError_t st = cudaGetDeviceCount(&ndev);
    if (st != cudaSuccess || ndev == 0)
        return fail(nullptr, MRB_E_CUDA, "mrb_create: no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(nullptr, MRB_E_ARG, "mrb_create: bad device index");
    cudaDeviceProp prop;
    if ((st = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return cuda_fail(nullptr, st, "cudaGetDeviceProperties");
    if (prop.major != 10)
        return fail(nullptr, MRB_E_UNSUPPORTED, "mrb_create: kernels are built for sm_100a (B200) only");

    mrb_env *e = new (std::nothrow) mrb_env();
    if (!e) return fail(nullptr, MRB_E_ARG, "mrb_create: out of host memory");
    // the scratch of mrb_step_masked, here so that no step allocates (a captured graph could not); the caller's
    // current device is left as it was
    int prev = device;
    cudaGetDevice(&prev);
    e->step_list = nullptr;
    if ((st = cudaSetDevice(device)) == cudaSuccess && (st = cudaMalloc(&e->step_list, sizeof(int32_t) * (num_envs + 3))) == cudaSuccess)
        st = cudaMemset(e->step_list + num_envs, 0, 3 * sizeof(int32_t));
    cudaSetDevice(prev);
    if (st != cudaSuccess) {
        if (e->step_list) cudaFree(e->step_list);
        delete e;
        return cuda_fail(nullptr, st, "mrb_create: step list");
    }
    std::memset(&e->p, 0, sizeof(Params));
    e->p.cfg = c;
    e->p.B = num_envs;
    e->p.env_lo = 0;
    e->p.env_hi = num_envs;
    e->p.env_id0 = env_id0;
    e->p.seed = 0;
    e->p.obs_dim = obs_dim_of(c);
    e->p.obs_blocks = obs_block_count(c);
    e->p.rows_f64 = rows_f64(c);
    e->p.rows_i32 = rows_i32(c);
    e->p.collision_thr2 = thr2(c.collision_diameter);
    e->p.sense_thr2 = thr2(c.predator_radius);
    e->p.capture_thr2 = thr2(c.capture_radius);
    e->p.zone1_thr2 = thr2(c.zone1_radius);
    e->device = device;
    e->bound = false;
    e->actions_dev = nullptr;
    e->pipe_ready = false;
    *out = e;
    return MRB_OK;
}

extern "C" int mrb_destroy(mrb_env *env)
{
    if (!env) return MRB_E_ARG;
    cudaSetDevice(env->device);
    if (env->actions_dev) cudaFree(env->actions_dev);
    if (env->step_list) cudaFree(env->step_list);
    if (env->pipe_ready) {
        for (int k = 0; k < kPipeStreams; k++) { cudaStreamDestroy(env->pipe[k]); cudaEventDestroy(env->ev_out[k]); }
        cudaEventDestroy(env->ev_in);
    }
    delete env;
    return MRB_OK;
}

static int num_actions_of(const mrb_config &c) { return c.scenario == MRB_MATERIAL ? 20 : 5; }

extern "C" int mrb_state_rows(const mrb_env *env, int32_t *rf, int32_t *ri)
{
    if (!env || !rf || !ri) return MRB_E_ARG;
    *rf = env->p.rows_f64; *ri = env->p.rows_i32;
    return MRB_OK;
}
extern "C" int mrb_obs_dim(const mrb_env *env) { return env ? env->p.obs_dim : MRB_E_ARG; }
extern "C" int mrb_num_actions(const mrb_env *env)
{
    if (!env) return MRB_E_ARG;
    return num_actions_of(env->p.cfg);     // spaces.Discrete(20) MaterialTransport.py:80, Discrete(5) elsewhere
}

extern "C" int mrb_bind(mrb_env *env, const mrb_buffers *b)
{
    if (!env || !b) return MRB_E_ARG;
    if (!b->state_f64 || !b->state_i32 || !b->obs || !b->reward || !b->done || !b->message || !b->remaining)
        return fail(env, MRB_E_ARG, "mrb_bind: state_f64, state_i32, obs, reward, done, message, remaining are required");
    if (env->p.cfg.track_dist && !b->dist) return fail(env, MRB_E_ARG, "mrb_bind: track_dist set but dist buffer is NULL");
    if (((uintptr_t)b->state_f64 | (uintptr_t)b->obs | (uintptr_t)b->reward) & 15)
        return fail(env, MRB_E_ARG, "mrb_bind: buffers must be 16-byte aligned");
    env->p.buf = *b;
    env->bound = true;
    return MRB_OK;
}

extern "C" int mrb_reset(mrb_env *env, const uint8_t *mask, uint64_t seed, void *stream)
{
    if (!env) return MRB_E_ARG;
    if (!env->bound) return fail(env, MRB_E_STATE, "mrb_reset: call mrb_bind first");
    cudaError_t st = cudaSetDevice(env->device);
    if (st != cudaSuccess) return cuda_fail(env, st, "cudaSetDevice");
    env->p.seed = seed;
    cudaStream_t s = (cudaStream_t)stream;
    if ((st = launch_reset(env->p, mask, s)) != cudaSuccess) return cuda_fail(env, st, "reset kernel launch");
    g_launches++;
    if ((st = cudaGetLastError()) != cudaSuccess) return cuda_fail(env, st, "reset kernel launch");
    return MRB_OK;
}

// launch the step kernel for envs [lo, hi) on stream s, or (list: env->step_list after the compaction) for the listed envs
static int step_range(mrb_env *env, const int32_t *actions, int64_t lo, int64_t hi, cudaStream_t s, const HostOut *hout = nullptr,
                      const int32_t *list = nullptr)
{
    Params p = env->p;
    p.env_lo = lo;
    p.env_hi = hi;
    if (hout) p.hout = *hout;
    if (list) { p.envs = list; p.count = list + p.B; }
    cudaError_t st;
    switch (p.cfg.scenario) {
    case MRB_PCP: st = launch_step<MRB_PCP>(p, actions, s); break;
    case MRB_WAREHOUSE: st = launch_step<MRB_WAREHOUSE>(p, actions, s); break;
    case MRB_MATERIAL: st = launch_step<MRB_MATERIAL>(p, actions, s); break;
    case MRB_ARCTIC: st = launch_step<MRB_ARCTIC>(p, actions, s); break;
    default: st = launch_step<MRB_SIMPLE>(p, actions, s); break;
    }
    if (st != cudaSuccess) return cuda_fail(env, st, "step kernel launch");
    g_launches++;
    if ((st = cudaGetLastError()) != cudaSuccess) return cuda_fail(env, st, "step kernel launch");
    return MRB_OK;
}

extern "C" int mrb_step(mrb_env *env, const int32_t *actions, void *stream)
{
    if (!env || !actions) return MRB_E_ARG;
    if (!env->bound) return fail(env, MRB_E_STATE, "mrb_step: call mrb_bind first");
    if ((uintptr_t)actions & 15) return fail(env, MRB_E_ARG, "mrb_step: actions must be 16-byte aligned");
    cudaError_t st = cudaSetDevice(env->device);
    if (st != cudaSuccess) return cuda_fail(env, st, "cudaSetDevice");
    return step_range(env, actions, 0, env->p.B, (cudaStream_t)stream);
}

// Two launches whatever `active` holds: the compaction into env->step_list, then the step kernel over the list, its grid
// sized for all B envs so that a captured graph does not depend on the mask.
extern "C" int mrb_step_masked(mrb_env *env, const int32_t *actions, const uint8_t *active, void *stream)
{
    if (!active) return mrb_step(env, actions, stream);
    if (!env) return MRB_E_ARG;
    if (!actions) return fail(env, MRB_E_ARG, "mrb_step_masked: actions is NULL");
    if (!env->bound) return fail(env, MRB_E_STATE, "mrb_step_masked: call mrb_bind first");
    if ((uintptr_t)actions & 15) return fail(env, MRB_E_ARG, "mrb_step_masked: actions must be 16-byte aligned");
    cudaPointerAttributes at;
    cudaError_t st = cudaPointerGetAttributes(&at, active);
    if (st != cudaSuccess) {
        cudaGetLastError();
        return fail(env, MRB_E_ARG, std::string("mrb_step_masked: active: ") + cudaGetErrorString(st));
    }
    if (at.type != cudaMemoryTypeDevice || at.device != env->device)
        return fail(env, MRB_E_ARG, "mrb_step_masked: active must be device memory of the env's device " + std::to_string(env->device));
    if ((st = cudaSetDevice(env->device)) != cudaSuccess) return cuda_fail(env, st, "cudaSetDevice");
    const cudaStream_t s = (cudaStream_t)stream;
    const int64_t B = env->p.B;
    if ((st = launch_compact(active, B, env->step_list, env->step_list + B, s)) != cudaSuccess)
        return cuda_fail(env, st, "compaction kernel launch");
    g_launches++;
    return step_range(env, actions, 0, B, s, nullptr, env->step_list);
}

// Host-buffer step.  Large batches are cut into up to 8 chunks, each on its own internal stream: all the
// (small) action uploads and all the chunk kernels are enqueued at once, so the kernels of several chunks
// share the SMs (a chunk of 8,192 envs fills a quarter of the machine and takes the same ~0.1 ms as a full
// wave) while the device->host copies - the PCIe-bound part: obs is 4*N*D bytes per env - drain chunk after
// chunk behind them on the copy engine.  Ordered after everything already enqueued on the caller's stream;
// synchronises before returning.
// Uploads, kernels and downloads of one chunked host step, forked from `s` onto the internal streams and joined
// back into `s`: pass 1 issues the upload + kernel of every chunk, pass 2 the downloads in chunk order.
// `small`: device aliases of the pinned reward / done / message buffers, or null.  When given, the kernel stores those
// three outputs straight into host memory and only the observations (94 % of the bytes) go through the copy engine:
// one download per chunk instead of four.
static int issue_host_step(mrb_env *env, const int32_t *actions_host, float *obs_host, float *reward_host,
                           uint8_t *done_host, uint8_t *message_host, int64_t chunk, cudaStream_t s, const HostOut *small)
{
    const int64_t B = env->p.B, N = env->p.cfg.num_robots, D = env->p.obs_dim;
    const mrb_buffers &b = env->p.buf;
    cudaError_t st;
    if ((st = cudaEventRecord(env->ev_in, s)) != cudaSuccess) return cuda_fail(env, st, "cudaEventRecord");
    int used = 0;
    for (int64_t lo = 0; lo < B; lo += chunk, used++) {
        const int64_t hi = lo + chunk < B ? lo + chunk : B, n = hi - lo;
        cudaStream_t ps = env->pipe[used];
        if ((st = cudaStreamWaitEvent(ps, env->ev_in, 0)) != cudaSuccess) return cuda_fail(env, st, "cudaStreamWaitEvent");
        if ((st = cudaMemcpyAsync(env->actions_dev + lo * N, actions_host + lo * N, sizeof(int32_t) * n * N, cudaMemcpyHostToDevice, ps)) != cudaSuccess)
            return cuda_fail(env, st, "H2D actions");
        const int rc = step_range(env, env->actions_dev, lo, hi, ps, small);
        if (rc != MRB_OK) return rc;
    }
    if (small) reward_host = nullptr, done_host = nullptr, message_host = nullptr;
    int k = 0;
    for (int64_t lo = 0; lo < B; lo += chunk, k++) {
        const int64_t hi = lo + chunk < B ? lo + chunk : B, n = hi - lo;
        cudaStream_t ps = env->pipe[k];
        if (obs_host && (st = cudaMemcpyAsync(obs_host + lo * N * D, b.obs + lo * N * D, sizeof(float) * n * N * D, cudaMemcpyDeviceToHost, ps)) != cudaSuccess)
            return cuda_fail(env, st, "D2H obs");
        if (reward_host && (st = cudaMemcpyAsync(reward_host + lo * N, b.reward + lo * N, sizeof(float) * n * N, cudaMemcpyDeviceToHost, ps)) != cudaSuccess)
            return cuda_fail(env, st, "D2H reward");
        if (done_host && (st = cudaMemcpyAsync(done_host + lo, b.done + lo, (size_t)n, cudaMemcpyDeviceToHost, ps)) != cudaSuccess)
            return cuda_fail(env, st, "D2H done");
        if (message_host && (st = cudaMemcpyAsync(message_host + lo, b.message + lo, (size_t)n, cudaMemcpyDeviceToHost, ps)) != cudaSuccess)
            return cuda_fail(env, st, "D2H message");
        if ((st = cudaEventRecord(env->ev_out[k], ps)) != cudaSuccess) return cuda_fail(env, st, "cudaEventRecord");
        if ((st = cudaStreamWaitEvent(s, env->ev_out[k], 0)) != cudaSuccess) return cuda_fail(env, st, "cudaStreamWaitEvent");
    }
    return MRB_OK;
}

static bool is_pinned_host(const void *ptr)
{
    if (!ptr) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

extern "C" int mrb_step_host(mrb_env *env, const int32_t *actions_host, float *obs_host, float *reward_host,
                             uint8_t *done_host, uint8_t *message_host, void *stream)
{
    if (!env || !actions_host) return MRB_E_ARG;
    if (!env->bound) return fail(env, MRB_E_STATE, "mrb_step_host: call mrb_bind first");
    cudaError_t st = cudaSetDevice(env->device);
    if (st != cudaSuccess) return cuda_fail(env, st, "cudaSetDevice");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t B = env->p.B, N = env->p.cfg.num_robots;
    if (!env->actions_dev && (st = cudaMalloc(&env->actions_dev, sizeof(int32_t) * B * N)) != cudaSuccess)
        return cuda_fail(env, st, "cudaMalloc(actions staging)");
    if (!env->pipe_ready) {
        for (int k = 0; k < kPipeStreams; k++) {
            if ((st = cudaStreamCreateWithFlags(&env->pipe[k], cudaStreamNonBlocking)) != cudaSuccess) return cuda_fail(env, st, "cudaStreamCreate");
            if ((st = cudaEventCreateWithFlags(&env->ev_out[k], cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(env, st, "cudaEventCreate");
        }
        if ((st = cudaEventCreateWithFlags(&env->ev_in, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(env, st, "cudaEventCreate");
        env->pipe_ready = true;
    }
    // chunk size: multiple of 64 envs keeps every chunk's actions 16-byte aligned; >= 16,384 envs per chunk
    int64_t nchunks = B / 16384;          // measured on B200 / PCIe 5: 65,536 PCP envs 0.61 / 0.53 / 0.53 / 0.58 / 0.68 ms at 1 / 2 / 4 / 8 / 16 chunks (direct issue)
    if (nchunks > 8) nchunks = 8;
    nchunks = nchunks < 1 ? 1 : (nchunks > kPipeStreams ? kPipeStreams : nchunks);
    int64_t chunk = (B + nchunks - 1) / nchunks;
    chunk = (chunk + 63) / 64 * 64;

    // Pinned buffers: the kernel can store into them through their device aliases (posted PCIe writes issued while it
    // runs).  Measured at 65,536 PCP envs: everything by copy engine 0.524 ms, everything by kernel stores 0.500 ms
    // (SM-issued writes reach ~38 GB/s against ~50 GB/s for the copy engine), hence the default split: the three small
    // outputs by kernel stores, the observations by one copy per chunk.  MRB_HOST_DIRECT=1 / 0 force all / nothing.
    static const int direct = [] { const char *e = std::getenv("MRB_HOST_DIRECT"); return e ? std::atoi(e) : -1; }();
    HostOut ho = {nullptr, nullptr, nullptr, nullptr};
    bool aliased = false;
    if (direct != 0) {
        const void *hp[4] = {obs_host, reward_host, done_host, message_host};
        void *dp[4] = {nullptr, nullptr, nullptr, nullptr};
        aliased = is_pinned_host(actions_host) && !((uintptr_t)obs_host & 15) && !((uintptr_t)reward_host & 3);
        for (int k = 0; k < 4 && aliased; k++)
            if (hp[k]) aliased = is_pinned_host(hp[k]) && cudaHostGetDevicePointer(&dp[k], const_cast<void *>(hp[k]), 0) == cudaSuccess;
        if (!aliased) cudaGetLastError();
        ho = {(float *)dp[0], (float *)dp[1], (uint8_t *)dp[2], (uint8_t *)dp[3]};
    }
    if (aliased && direct == 1) {
        if ((st = cudaMemcpyAsync(env->actions_dev, actions_host, sizeof(int32_t) * B * N, cudaMemcpyHostToDevice, s)) != cudaSuccess)
            return cuda_fail(env, st, "H2D actions");
        const int rc = step_range(env, env->actions_dev, 0, B, s, &ho);
        if (rc != MRB_OK) return rc;
        if ((st = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_fail(env, st, "mrb_step_host sync");
        return MRB_OK;
    }
    ho.obs = nullptr;
    const int rc = issue_host_step(env, actions_host, obs_host, reward_host, done_host, message_host, chunk, s, aliased ? &ho : nullptr);
    if (rc != MRB_OK) return rc;
    if ((st = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_fail(env, st, "mrb_step_host sync");
    return MRB_OK;
}

extern "C" int mrb_barrier_qp(int device, int32_t N, int32_t barrier_default, int64_t B, const double *dxi,
                              const double *xi, double *u, int32_t *iters, void *stream)
{
    if (!dxi || !xi || !u || B < 1 || N < 1 || N > MRB_MAX_ROBOTS) return fail(nullptr, MRB_E_ARG, "mrb_barrier_qp: bad argument");
    cudaError_t st = cudaSetDevice(device);
    if (st != cudaSuccess) return cuda_fail(nullptr, st, "cudaSetDevice");
    cudaStream_t s = (cudaStream_t)stream;
    if ((st = launch_barrier_qp(N, barrier_default, B, dxi, xi, u, iters, s)) != cudaSuccess) return cuda_fail(nullptr, st, "qp kernel launch");
    g_launches++;
    if ((st = cudaGetLastError()) != cudaSuccess) return cuda_fail(nullptr, st, "qp kernel launch");
    return MRB_OK;
}

extern "C" int mrb_select_actions(int device, int64_t num_envs, int32_t n_agents, int32_t n_actions,
                                  const mrb_select_desc *desc, int64_t *step, const float *q, int32_t *actions,
                                  void *stream)
{
    if (!desc || !step || !actions) return fail(nullptr, MRB_E_ARG, "mrb_select_actions: desc, step and actions are required");
    if (desc->struct_size != (int32_t)sizeof(mrb_select_desc))
        return fail(nullptr, MRB_E_ARG, "mrb_select_actions: mrb_select_desc.struct_size does not match this library (ABI mismatch)");
    if (desc->mode != MRB_SELECT_EPSILON_GREEDY && desc->mode != MRB_SELECT_SOFTMAX)
        return fail(nullptr, MRB_E_ARG, "mrb_select_actions: unknown mode");
    if (num_envs < 1 || n_agents < 1 || n_actions < 1)
        return fail(nullptr, MRB_E_ARG, "mrb_select_actions: num_envs, n_agents and n_actions must be >= 1");
    if (num_envs > ((int64_t)1 << 39) / n_agents)        // one 256-thread CTA per 256 rows: at most 2^31 CTAs
        return fail(nullptr, MRB_E_ARG, "mrb_select_actions: num_envs * n_agents must be <= 2^39");
    if (!(desc->eps_start >= 0.0 && desc->eps_start <= 1.0 && desc->eps_finish >= 0.0 && desc->eps_finish <= 1.0))
        return fail(nullptr, MRB_E_ARG, "mrb_select_actions: eps_start and eps_finish must be in [0, 1]");
    if (desc->anneal_time < 1) return fail(nullptr, MRB_E_ARG, "mrb_select_actions: anneal_time must be >= 1");
    if (desc->mode == MRB_SELECT_SOFTMAX && !q) return fail(nullptr, MRB_E_ARG, "mrb_select_actions: softmax needs q");
    cudaError_t st = cudaSetDevice(device);
    if (st != cudaSuccess) return cuda_fail(nullptr, st, "cudaSetDevice");
    st = launch_select_actions(num_envs, n_agents, n_actions, *desc, step, q, actions, (cudaStream_t)stream);
    if (st != cudaSuccess) return cuda_fail(nullptr, st, "select kernel launch");
    g_launches += 2;
    return MRB_OK;
}

// Everything mrb_record_begin / mrb_record_step check before they touch the device.
static int check_episode_batch(mrb_env *env, const mrb_episode_batch *b, const char *fn)
{
    const std::string f(fn);
    if (!env) return fail(nullptr, MRB_E_ARG, f + ": env is NULL");
    if (!b) return fail(env, MRB_E_ARG, f + ": batch is NULL");
    if (b->struct_size != (int32_t)sizeof(mrb_episode_batch))
        return fail(env, MRB_E_ARG, f + ": mrb_episode_batch.struct_size does not match this library (ABI mismatch)");
    if (!b->obs || !b->state || !b->actions || !b->actions_onehot || !b->avail_actions || !b->reward || !b->terminated ||
        !b->filled || !b->cursor)
        return fail(env, MRB_E_ARG, f + ": every pointer of mrb_episode_batch is required");
    if (b->state != b->obs) return fail(env, MRB_E_ARG, f + ": state must be obs (state = concat(obs), the same memory)");
    if (b->episode_limit < 1 || b->episode_limit > (1 << 30))
        return fail(env, MRB_E_ARG, f + ": episode_limit must be in [1, 2^30]");
    if (b->obs_width < env->p.obs_dim || b->obs_width > 65536)
        return fail(env, MRB_E_ARG, f + ": obs_width must be in [obs_dim, 65536]");
    // the kernel's accesses are scalar, each at its element's width
    if ((((uintptr_t)b->actions | (uintptr_t)b->filled) & 7) ||
        (((uintptr_t)b->obs | (uintptr_t)b->actions_onehot | (uintptr_t)b->avail_actions | (uintptr_t)b->reward |
          (uintptr_t)b->cursor) & 3))
        return fail(env, MRB_E_ARG, f + ": actions and filled must be 8-byte aligned, obs, actions_onehot, avail_actions, "
                                        "reward and cursor 4-byte aligned");
    if (!env->bound) return fail(env, MRB_E_STATE, f + ": call mrb_bind first");
    return MRB_OK;
}

static int record(mrb_env *env, const mrb_episode_batch *b, bool begin, const int32_t *actions, void *stream)
{
    cudaError_t st = cudaSetDevice(env->device);
    if (st != cudaSuccess) return cuda_fail(env, st, "cudaSetDevice");
    if ((st = launch_record(env->p, num_actions_of(env->p.cfg), *b, begin, actions, (cudaStream_t)stream)) != cudaSuccess)
        return cuda_fail(env, st, "record kernel launch");
    g_launches++;
    return MRB_OK;
}

extern "C" int mrb_record_begin(mrb_env *env, const mrb_episode_batch *batch, void *stream)
{
    const int rc = check_episode_batch(env, batch, "mrb_record_begin");
    return rc != MRB_OK ? rc : record(env, batch, true, nullptr, stream);
}

extern "C" int mrb_record_step(mrb_env *env, const mrb_episode_batch *batch, const int32_t *actions, void *stream)
{
    int rc = check_episode_batch(env, batch, "mrb_record_step");
    if (rc != MRB_OK) return rc;
    if (!actions || ((uintptr_t)actions & 3)) return fail(env, MRB_E_ARG, "mrb_record_step: actions must be a 4-byte aligned device pointer");
    return record(env, batch, false, actions, stream);
}

// Everything mrb_eval_begin / mrb_eval_step check before they touch the device.
static int check_eval_table(mrb_env *env, const mrb_eval_table *t, const char *fn)
{
    const std::string f(fn);
    if (!env) return fail(nullptr, MRB_E_ARG, f + ": env is NULL");
    if (!t) return fail(env, MRB_E_ARG, f + ": table is NULL");
    if (t->struct_size != (int32_t)sizeof(mrb_eval_table))
        return fail(env, MRB_E_ARG, f + ": mrb_eval_table.struct_size does not match this library (ABI mismatch)");
    if (!t->return_ || !t->length || !t->message || !t->timeout || !t->remaining || !t->dist || !t->acc_return ||
        !t->acc_length || !t->acc_dist || !t->count)
        return fail(env, MRB_E_ARG, f + ": every pointer of mrb_eval_table is required");
    if (t->episodes < 1 || t->episodes > (1 << 20)) return fail(env, MRB_E_ARG, f + ": episodes must be in [1, 2^20]");
    // the kernel's accesses are scalar, each at its element's width
    if ((((uintptr_t)t->return_ | (uintptr_t)t->acc_return | (uintptr_t)t->acc_dist) & 7) ||
        (((uintptr_t)t->length | (uintptr_t)t->remaining | (uintptr_t)t->dist | (uintptr_t)t->acc_length |
          (uintptr_t)t->count) & 3))
        return fail(env, MRB_E_ARG, f + ": return_, acc_return and acc_dist must be 8-byte aligned, length, remaining, "
                                        "dist, acc_length and count 4-byte aligned");
    if (!env->bound) return fail(env, MRB_E_STATE, f + ": call mrb_bind first");
    return MRB_OK;
}

static int eval(mrb_env *env, const mrb_eval_table *t, bool begin, void *stream)
{
    const int rc = check_eval_table(env, t, begin ? "mrb_eval_begin" : "mrb_eval_step");
    if (rc != MRB_OK) return rc;
    cudaError_t st = cudaSetDevice(env->device);
    if (st != cudaSuccess) return cuda_fail(env, st, "cudaSetDevice");
    if ((st = launch_eval(env->p, *t, begin, (cudaStream_t)stream)) != cudaSuccess)
        return cuda_fail(env, st, "eval kernel launch");
    g_launches++;
    return MRB_OK;
}

extern "C" int mrb_eval_begin(mrb_env *env, const mrb_eval_table *table, void *stream) { return eval(env, table, true, stream); }

extern "C" int mrb_eval_step(mrb_env *env, const mrb_eval_table *table, void *stream) { return eval(env, table, false, stream); }
