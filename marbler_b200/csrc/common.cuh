// Shared device-side definitions for the marbler_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "../../include/marbler_b200.h"

namespace mrb {

// rps RobotariumABC constants (SURVEY.md App. A.1) -- the ones flagged "(?)" there are named here
// so that a correction against rps@6bb184e is a one-line change.
constexpr double kTimeStep = 0.033;
constexpr double kMaxLinearVelocity = 0.2;
constexpr double kMaxAngularVelocity = 2.0 * (0.016 / 0.11) * (0.2 / 0.016);
constexpr double kArenaXMin = -1.6, kArenaXMax = -1.6 + 3.2, kArenaYMin = -1.0, kArenaYMax = -1.0 + 2.0;
// controller constants (App. A.6 - A.8)
constexpr double kProjectionDistance = 0.05;
constexpr double kSiVelocityLimit = 0.15;
constexpr double kAngularLimit = 3.14159265358979323846;
constexpr double kQpMagnitudeLimit = 0.2;
constexpr double kPi = 3.14159265358979323846;
constexpr double kTwoPi = 6.28318530717958647692;

// Host mirrors of the step outputs (mrb_step_host): device-visible aliases of the caller's pinned buffers.  When
// set, the step kernel stores obs / reward / done / message there as well, so the results cross PCIe as posted
// writes while the kernel is still running instead of in copy-engine transfers queued behind it.
struct HostOut {
    float *obs, *reward;
    uint8_t *done, *message;
};

// Everything a kernel needs, passed by value (__grid_constant__).
struct Params {
    mrb_config cfg;
    mrb_buffers buf;
    HostOut hout;       // all null outside the direct host path
    int64_t B;          // envs on this device (row stride of the state arrays)
    int64_t env_lo, env_hi;   // this launch processes envs [env_lo, env_hi)
    int64_t env_id0;    // global id of env 0 (RNG stream offset of this rank)
    uint64_t seed;
    int32_t obs_dim;    // D
    int32_t obs_blocks; // neighbour blocks per agent incl. self (PCP / Warehouse)
    int32_t rows_f64, rows_i32;
    // exact squared thresholds: sqrt(d2) <= r  <=>  d2 <= thr2(r)   (computed on the host)
    double collision_thr2, sense_thr2, capture_thr2, zone1_thr2;
    // mrb_step_masked: the compacted ids of the active envs and their number (written by the compaction kernel on the
    // stream); item i of the step launch steps env envs[i] and items >= *count none.  NULL on every other path.
    const int32_t *envs, *count;
};

// ---- state rows (env index fastest).  f64 rows:
//   [0,N) x | [N,2N) y | [2N,3N) theta | [3N,4N) prev x | [4N,5N) prev y | 5N: episode return |
//   5N+1 ..: scenario rows (PCP prey x0,y0,x1,y1,...; Simple goal x,y)
// i32 rows: 0 episode_steps | 1 prev_valid | 2 episode_count | 3.. scenario rows
//   PCP: sensed mask, captured mask | Warehouse: loaded mask |
//   MaterialTransport: load[N], zone1, zone2, messages (2 bits each) |
//   ArcticTransport: grid (6 words, 2 bits per cell, cell = row*12+col), goal_col, pixel_type (2 bits each), reached mask
__host__ __device__ inline int scenario_rows_f64(const mrb_config &c)
{
    return c.scenario == MRB_PCP ? 2 * c.num_prey : (c.scenario == MRB_SIMPLE ? 2 : 0);
}
__host__ __device__ inline int scenario_rows_i32(const mrb_config &c)
{
    switch (c.scenario) {
    case MRB_PCP: return 2;
    case MRB_WAREHOUSE: return 1;
    case MRB_MATERIAL: return c.num_robots + 3;
    case MRB_ARCTIC: return 9;
    default: return 0;
    }
}
__host__ __device__ inline int rows_f64(const mrb_config &c) { return 5 * c.num_robots + 1 + scenario_rows_f64(c); }
constexpr int kCommonRowsI32 = 3;
__host__ __device__ inline int rows_i32(const mrb_config &c) { return kCommonRowsI32 + scenario_rows_i32(c); }

// ---- Philox4x32-10 (Salmon et al. SC'11); key = seed, counter = (env id, episode, block)
struct Philox {
    uint32_t key0, key1, c0, c1, c2, c3, buf[4];
    int have;
    __device__ Philox(uint64_t seed, uint64_t env_id, uint32_t episode)
        : key0((uint32_t)seed), key1((uint32_t)(seed >> 32)), c0((uint32_t)env_id), c1((uint32_t)(env_id >> 32)),
          c2(episode), c3(0), have(0) {}
    __device__ void refill()
    {
        uint32_t a0 = c0, a1 = c1, a2 = c2, a3 = c3, k0 = key0, k1 = key1;
#pragma unroll
        for (int r = 0; r < 10; r++) {
            uint32_t hi0 = __umulhi(0xD2511F53u, a0), lo0 = 0xD2511F53u * a0;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, a2), lo1 = 0xCD9E8D57u * a2;
            uint32_t n0 = hi1 ^ a1 ^ k0, n2 = hi0 ^ a3 ^ k1;
            a0 = n0; a1 = lo1; a2 = n2; a3 = lo0;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        buf[0] = a0; buf[1] = a1; buf[2] = a2; buf[3] = a3;
        c3++;
        have = 4;
    }
    __device__ uint32_t u32()
    {
        if (!have) refill();
        uint32_t v = have == 4 ? buf[0] : (have == 3 ? buf[1] : (have == 2 ? buf[2] : buf[3]));
        have--;
        return v;
    }
    __device__ uint32_t below(uint32_t n) { return __umulhi(u32(), n); }
    __device__ double unit()
    {
        uint32_t a = u32() >> 5, b = u32() >> 6;
        return (a * 67108864.0 + b) / 9007199254740992.0;
    }
    __device__ double normal()
    {
        double u1 = 1.0 - unit(), u2 = unit();
        return sqrt(-2.0 * log(u1)) * cos(2.0 * kPi * u2);
    }
};

// compile-time loop: f(std::integral_constant<int, I>) for I in [B, E).  nvcc's `#pragma unroll` gives up
// on triangular loop nests (it leaves a runtime loop and the factor lands in local memory); with the
// outer index a template constant every inner bound is a literal and unrolls reliably.
template <int B, int E, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (B < E) {
        f(std::integral_constant<int, B>{});
        static_for<B + 1, E>(f);
    }
}

// 1/x without the IEEE fix-up path: MUFU seed + two Newton steps (relative error ~1e-16)
__device__ __forceinline__ double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}
// one Newton step only: relative error ~2^-46 (1.4e-14).  Used where the value only scales a Newton
// direction or a step length (the iteration recomputes its residuals, so this does not accumulate).
__device__ __forceinline__ double fast_rcp1(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    return fma(r, e, r);
}
__device__ __forceinline__ double fast_rsqrt(double x)
{
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double hx = 0.5 * x;
    r = r * fma(-hx * r, r, 1.5);
    r = r * fma(-hx * r, r, 1.5);
    return r;
}

__device__ __forceinline__ double clampd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }
// sin and cos of a small angle (|x| <= 0.125; the step kernels pass dt * omega, |.| <= 0.12): Taylor polynomials in
// x^2, truncation error < 2^-53 relative - a dozen FMAs instead of the library's range reduction
__device__ __forceinline__ void small_sincos(double x, double &s, double &c)
{
    const double x2 = x * x;
    double ps = fma(x2, 1.0 / 362880.0, -1.0 / 5040.0);
    ps = fma(ps, x2, 1.0 / 120.0);
    ps = fma(ps, x2, -1.0 / 6.0);
    s = fma(x * x2, ps, x);
    double pc = fma(x2, -1.0 / 3628800.0, 1.0 / 40320.0);
    pc = fma(pc, x2, -1.0 / 720.0);
    pc = fma(pc, x2, 1.0 / 24.0);
    pc = fma(pc, x2, -0.5);
    c = fma(pc, x2, 1.0);
}

// sin and cos of a heading (|x| <= 4; the step kernels pass theta in (-pi, pi]): quadrant by a two-term Cody-Waite
// reduction (exact enough for |k| <= 3), then the fdlibm kernel polynomials on [-pi/4, pi/4].  Error <= 1 ulp
// (2.2e-16 against libm over [-4, 4], checked on the host); ~35 instructions against ~130 for the library's sincos with
// its large-argument path.
__device__ __forceinline__ void heading_sincos(double x, double &s, double &c)
{
    const double kd = rint(x * 0.63661977236758134308);                     // 2 / pi
    const int k = (int)kd;
    double r = fma(-kd, 1.57079632679489655800e+00, x);
    r = fma(-kd, 6.12323399573676603587e-17, r);
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(ps, z, 2.75573137070700676789e-06);
    ps = fma(ps, z, -1.98412698298579493134e-04);
    ps = fma(ps, z, 8.33333333332248946124e-03);
    ps = fma(ps, z, -1.66666666666666324348e-01);
    const double sr = fma(r * z, ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(pc, z, -2.75573143513906633035e-07);
    pc = fma(pc, z, 2.48015872894767294178e-05);
    pc = fma(pc, z, -1.38888888888741095749e-03);
    pc = fma(pc, z, 4.16666666666666019037e-02);
    const double cr = fma(z * z, pc, fma(-0.5, z, 1.0));
    const bool swap = k & 1;
    const double a = swap ? cr : sr, b = swap ? sr : cr;
    s = (k & 2) ? -a : a;
    c = ((k + 1) & 2) ? -b : b;
}

// max / min as compare + select: 3 instructions.  fmax / fmin carry IEEE NaN handling that costs 7 (DSETP.MAX, three
// moves, FSEL, SEL, LOP3) - measured at 27 of them per interior-point iteration, a fifth of the loop body.  A NaN in
// `a` is dropped (the comparison is false), which is all the solvers need: tmax = dmax(candidate, tmax).
__device__ __forceinline__ double dmax(double a, double b) { return a > b ? a : b; }
__device__ __forceinline__ double dmin(double a, double b) { return a < b ? a : b; }
// maximum of M candidates by a pairwise tree: depth log2(M) instead of a serial chain of M dependent selects (a
// compare + select is ~13 cycles of latency, and the one-env-per-thread kernels run 2 warps per scheduler)
template <int M>
__device__ __forceinline__ double tree_max(double (&v)[M])
{
#pragma unroll
    for (int s = 1; s < M; s *= 2)
#pragma unroll
        for (int i = 0; i + s < M; i += 2 * s) v[i] = dmax(v[i + s], v[i]);
    return v[0];
}

// ---- one weight set of mrb_policy_create / mrb_policy_load: state_dict order, torch layout ([out][in] row-major)
// (include/marbler_b200.h).  Without a GRU, wih / bih are rnn.weight / rnn.bias and whh / bhh are unused.
__host__ __device__ inline int64_t weight_set_floats(int H, int Din, int A, bool rnn)
{
    return (int64_t)H * Din + H + (rnn ? 2LL * 3 * H * H + 2 * 3 * H : (int64_t)H * H + H) + (int64_t)A * H + A;
}
struct WeightSet {
    const float *fc1w, *fc1b, *wih, *whh, *bih, *bhh, *fc2w, *fc2b;
    __host__ __device__ WeightSet(const float *w, int H, int Din, int A, bool rnn)
    {
        fc1w = w; fc1b = fc1w + (size_t)H * Din; wih = fc1b + H;
        if (rnn) { whh = wih + (size_t)3 * H * H; bih = whh + (size_t)3 * H * H; bhh = bih + 3 * H; fc2w = bhh + 3 * H; }
        else { whh = nullptr; bih = wih + (size_t)H * H; bhh = nullptr; fc2w = bih + H; }
        fc2b = fc2w + (size_t)A * H;
    }
};

}  // namespace mrb
