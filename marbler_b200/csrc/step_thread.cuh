// One environment per thread: the whole MARBLER env step (goal generation, UF sub-steps of
// controller + barrier QP + unicycle integration + violation checks, scenario events / observations
// / rewards / done, optional auto-reset) between one coalesced read and one write of the SoA state.
//
// Reference call stack being replaced (SURVEY.md 3.3, App. C):
//   wrapper.py:41-44 Wrapper.step -> <Scenario>.step -> utilities/roboEnv.py:38-96 roboEnv.step
//   -> utilities/controller.py:20-25 -> rps (App. A.2-A.8) -> cvxopt.solvers.qp (A.9)
#pragma once
#include "common.cuh"
#include "qp_thread.cuh"
#include "qp_dual.cuh"

namespace mrb {

// CTA shape, from the measurements in DESIGN.md section 4.  Teams of up to 4 robots (dual QP, everything in registers):
// 255 registers and 64-thread CTAs, 4 per SM (32- and 128-thread CTAs measured the same, every lower register cap
// slower).  Teams of 5 and 6 robots (primal QP): the shape is set by the shared-memory QP store, not by registers --
// one 8-warp CTA per SM, whose warps run the 12 k-instruction body in step and share the instruction fetches.
template <int N>
struct ThreadShape {
    static constexpr bool kPrimal = !(N >= 2 && N <= 4);     // up to 4 robots the dual Newton system is the smaller one (m <= 6 < 2N)
    static constexpr int kThreads = kPrimal ? 256 : 64;
    static constexpr int kMinBlocks = kPrimal ? 1 : 4;
};

// Per-CTA shared store of the primal QP (qp_thread.cuh): [factor words (double2) | h, rz (double)], interleaved over
// the threads.  The dual QP has none: its teams launch with 0 bytes of dynamic shared memory.
template <int N, bool = ThreadShape<N>::kPrimal>
struct QpStore {
    static constexpr size_t kBytes = 0;
};
template <int N>
struct QpStore<N, true> {
    using Qp = QpThread<N, ThreadShape<N>::kThreads>;
    static constexpr size_t kBytes = (size_t)(Qp::kSmemWords + Qp::kVecDoubles / 2) * ThreadShape<N>::kThreads * sizeof(double2);
    double2 *Ls;
    double *Vs;
    __device__ __forceinline__ QpStore()
    {
        extern __shared__ double2 store[];           // kBytes, sized by the launcher
        Ls = store + threadIdx.x;
        Vs = reinterpret_cast<double *>(store + Qp::kSmemWords * ThreadShape<N>::kThreads) + threadIdx.x;
    }
};
static_assert(QpStore<5>::kBytes == 122880 && QpStore<6>::kBytes == 184320, "primal QP store: 120 / 180 KB per CTA");

template <int N>
__device__ __forceinline__ int qp_run(const double (&xix)[N], const double (&xiy)[N], double (&ux)[N], double (&uy)[N],
                                      bool barrier_default, const QpStore<N> &st)
{
    if constexpr (ThreadShape<N>::kPrimal) {
        typename QpStore<N>::Qp qp(st.Ls, st.Vs);
        return qp.run(xix, xiy, ux, uy, barrier_default);
    } else {
        QpDual<N> qp;
        return qp.run(xix, xiy, ux, uy, barrier_default);
    }
}

// every scenario's Agent.generate_goal: PredatorCapturePrey/agent.py:48-76, warehouse.py:19-45,
// MaterialTransport.py:19-46, ArcticTransport/agent.py:114-137, simple.py:32-60
__device__ __forceinline__ void generate_goal(const mrb_config &c, double step, int action, double x, double y,
                                              double &gx, double &gy)
{
    const double cx = x < c.left ? c.left : (x > c.right ? c.right : x);
    const double cy = y < c.up ? c.up : (y > c.down ? c.down : y);
    gx = cx; gy = cy;
    if (action == 0) gx = fmax(x - step, c.left);
    else if (action == 1) gx = fmin(x + step, c.right);
    else if (action == 2) gy = fmax(y - step, c.up);
    else if (action == 3) gy = fmin(y + step, c.down);
}

template <int SCN, int N>
__device__ __forceinline__ double agent_step_size(const mrb_config &c, int i, int pixel_types)
{
    if (SCN == MRB_MATERIAL) return i < c.n_fast ? c.fast_step : c.slow_step;       // MaterialTransport.py:71-74
    if (SCN == MRB_ARCTIC) {                                                          // ArcticTransport/agent.py:94-112
        if (i < 2) return c.fast_step;
        const int p = (pixel_types >> (2 * i)) & 3;
        if (i == 3) return p == 1 ? c.slow_step : (p == 2 ? c.fast_step : c.step_dist);
        return p == 1 ? c.fast_step : (p == 2 ? c.slow_step : c.step_dist);
    }
    return c.step_dist;
}

// utilities/misc.py:23 np.linalg.norm(poses[:2,x]-poses[:2,agent]): the K-nearest order is decided on the
// ROUNDED norm (near-ties on the spawn grid are common), so no FMA contraction and a real sqrt here
__device__ __forceinline__ double neighbor_dist(double dx, double dy)
{
    return __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

// ArcticTransport.py:136-143 get_cell_from_pose (int() truncates toward zero)
__device__ __forceinline__ void arctic_cell(double x, double y, int &row, int &col)
{
    int r = -(int)((y - 1.0) / .25), cc = (int)((x + 1.5) / .25);
    row = r < 0 ? 0 : (r > 7 ? 7 : r);
    col = cc < 0 ? 0 : (cc > 11 ? 11 : cc);
}
__device__ __forceinline__ int arctic_grid(const uint32_t (&g)[6], int row, int col)
{
    const int k = row * 12 + col, wi = k >> 4;
    uint32_t w = g[0];
#pragma unroll
    for (int t = 1; t < 6; t++) w = (wi == t) ? g[t] : w;
    return (w >> (2 * (k & 15))) & 3;
}

// one agent's observation row: float32 always, plus the optional float64 copy (mrb_buffers.obs_f64)
struct ObsRow {
    float *f;
    double *d;
    __device__ __forceinline__ ObsRow(float *f_, double *d64, int64_t off) : f(f_ + off), d(d64 ? d64 + off : nullptr) {}
    __device__ __forceinline__ void put(int k, double v) const
    {
        f[k] = (float)v;
        if (d) d[k] = v;
    }
};

// ---- reset: <Scenario>.reset() + roboEnv.reset() (distributional parity, SURVEY 8a row a14)
// index of the r-th (0-based) set bit of m: five popcount steps instead of a scan over the cells (the reset path runs
// with one active lane per warp inside the step kernel, so its cost is its dependent instruction count)
__device__ __forceinline__ int nth_set_bit(uint32_t m, int r)
{
    int pos = 0;
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
        const int c = __popc(m & ((1u << w) - 1u));
        if (r >= c) { r -= c; m >>= w; pos += w; }
    }
    return pos;
}
// N distinct cells of the spawn grid, uniformly, in order (rps generate_initial_conditions, App. A.5): draw i takes the
// r-th still-free cell in ascending order, r uniform in [0, cells - i)
template <typename F>
__device__ __forceinline__ void spawn_grid(const mrb_spawn &sp, Philox &g, F emit)
{
    const int cells = sp.xr * sp.yr;
    uint64_t freem = cells >= 64 ? ~0ull : ((1ull << cells) - 1ull);
    // cell / yr for cell < 64 as a multiply-shift (exact for every yr in 1..64: checked exhaustively in tests/test_host_logic.py)
    const uint32_t inv = (65536u + (uint32_t)sp.yr - 1u) / (uint32_t)sp.yr;
    for (int i = 0; i < sp.count; i++) {
        int r = (int)g.below((uint32_t)(cells - i));
        const uint32_t lo = (uint32_t)freem, hi = (uint32_t)(freem >> 32);
        const int nlo = __popc(lo);
        const int cell = r < nlo ? nth_set_bit(lo, r) : 32 + nth_set_bit(hi, r - nlo);
        freem &= ~(1ull << cell);
        const int ix = (int)(((uint32_t)cell * inv) >> 16), iy = cell - ix * sp.yr;
        // explicit _rn ops: no FMA contraction, so the spawn poses are bit-identical to numpy's
        const double x = __dadd_rn(__dadd_rn(__dsub_rn(__dmul_rn((double)ix, sp.spacing), sp.w2), sp.sx1), sp.sx2);
        const double y = __dadd_rn(__dadd_rn(__dsub_rn(__dmul_rn((double)iy, sp.spacing), sp.h2), sp.sy1), sp.sy2);
        double th = 0.0;
        if (sp.random_theta) {                       // warehouse.py:93 keeps rps' random heading
            th = g.unit() * kTwoPi - kPi;
            th = atan2(sin(th), cos(th));            // the zero-velocity sim step of roboEnv.py:112
        }
        emit(i, x, y, th);
    }
}

// `episode`: the env's episode counter (state_i32 row 2), read by the caller - the step kernels fetch it while their
// write-back is in flight instead of stalling on it here
template <int SCN>
__device__ void reset_env(const Params &p, int64_t env, int32_t episode)
{
    const mrb_config &c = p.cfg;
    const int N = c.num_robots;
    const int64_t S = p.B;
    double *sf = p.buf.state_f64 + env;
    int32_t *si = p.buf.state_i32 + env;
    Philox g(p.seed, (uint64_t)(p.env_id0 + env), (uint32_t)episode);
    si[0] = 0;
    si[1 * S] = 0;
    si[2 * S] = episode + 1;
    for (int r = 3 * N; r < 5 * N + 1; r++) sf[r * S] = 0.0;       // prev pose, episode return
    int32_t *sci = si + kCommonRowsI32 * S;
    double *scf = sf + (5 * N + 1) * S;
    if (SCN == MRB_ARCTIC) {                                        // ArcticTransport.py:28-33, 56-82
        const double sx[4] = {-.3, .3, -.9, .9};
        for (int i = 0; i < N; i++) {
            sf[i * S] = sx[i & 3];
            sf[(N + i) * S] = -.8;
            sf[(2 * N + i) * S] = atan2(sin(kPi / 2), cos(kPi / 2));
        }
        uint32_t w[6] = {0, 0, 0, 0, 0, 0};
        for (int k = 0; k < 96; k++) w[k >> 4] |= g.below(3) << (2 * (k & 15));
        const int gc = 1 + (int)g.below(11);
        for (int k = 1; k < 11; k++) w[(84 + k) >> 4] &= ~(3u << (2 * ((84 + k) & 15)));
        const int goal_cells[4] = {gc, gc - 1, 12 + gc, 12 + gc - 1};
        for (int t = 0; t < 4; t++) w[goal_cells[t] >> 4] |= 3u << (2 * (goal_cells[t] & 15));
        for (int t = 0; t < 6; t++) sci[t * S] = (int32_t)w[t];
        sci[6 * S] = gc;
        sci[7 * S] = 0;
        sci[8 * S] = 0;
        return;
    }
    spawn_grid(c.spawn_robots, g, [&](int i, double x, double y, double th) {
        sf[i * S] = x; sf[(N + i) * S] = y; sf[(2 * N + i) * S] = th;
    });
    if (SCN == MRB_PCP) {                                           // PredatorCapturePrey.py:128-132
        spawn_grid(c.spawn_other, g, [&](int i, double x, double y, double) {
            scf[(2 * i) * S] = x; scf[(2 * i + 1) * S] = y;
        });
        sci[0] = 0; sci[S] = 0;
    } else if (SCN == MRB_SIMPLE) {                                 // simple.py:141-144
        spawn_grid(c.spawn_other, g, [&](int, double x, double y, double) { scf[0] = x; scf[S] = y; });
    } else if (SCN == MRB_WAREHOUSE) {
        sci[0] = 0;
    } else if (SCN == MRB_MATERIAL) {                               // MaterialTransport.py:96-103
        for (int i = 0; i < N; i++) sci[i * S] = 0;
        for (int k = 0; k < 2; k++) sci[(N + k) * S] = (int32_t)(c.zone_mu[k] + c.zone_sigma[k] * g.normal());
        sci[(N + 2) * S] = 0;
    }
}

template <int SCN>
__global__ void reset_kernel(const __grid_constant__ Params p, const uint8_t *mask)
{
    const int64_t env = p.env_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.env_hi) return;
    if (mask && !mask[env]) return;
    reset_env<SCN>(p, env, p.buf.state_i32[env + 2 * p.B]);
    // the reference returns an all-zero observation from reset (e.g. PredatorCapturePrey.py:136)
    const int nd = p.cfg.num_robots * p.obs_dim;
    float *o = p.buf.obs + env * nd;
    for (int k = 0; k < nd; k++) o[k] = 0.f;
    if (p.buf.obs_f64)
        for (int k = 0; k < nd; k++) p.buf.obs_f64[env * nd + k] = 0.0;
}

// ---- the step
// LIST = {true} (mrb_step_masked): item i steps env p.envs[i]; the live items are a prefix of the launch, so the warps
// are full but for the last one.  LIST empty: item i steps env env_lo + i.  A compile-time switch, because read at run
// time the env index could no longer be recomputed from blockIdx where registers are short (the N = 4 kernel would
// spill); an empty pack, so that the range kernels keep their names and their code.
template <int SCN, int N, bool... LIST>
__global__ void __launch_bounds__(ThreadShape<N>::kThreads, ThreadShape<N>::kMinBlocks)
step_thread_kernel(const __grid_constant__ Params p, const int32_t *__restrict__ actions)
{
    constexpr bool kList = (false || ... || LIST);
    const int64_t item = (int64_t)blockIdx.x * ThreadShape<N>::kThreads + threadIdx.x;
    const int64_t env = kList ? (item < *p.count ? (int64_t)p.envs[item] : -1) : p.env_lo + item;
    const bool live = kList ? env >= 0 : env < p.env_hi;
    const unsigned warp_envs = __ballot_sync(0xffffffffu, live);      // lanes of this warp that own an env
    if (!live) return;
    const mrb_config &c = p.cfg;
    const int64_t S = p.B;
    double *sf = p.buf.state_f64 + env;
    int32_t *si = p.buf.state_i32 + env;
    int32_t *sci = si + kCommonRowsI32 * S;
    double *scf = sf + (5 * N + 1) * S;
    const QpStore<N> qp_smem;

    double px[N], py[N], th[N], qx[N], qy[N];
    int act[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
        px[i] = sf[i * S]; py[i] = sf[(N + i) * S]; th[i] = sf[(2 * N + i) * S];
        qx[i] = sf[(3 * N + i) * S]; qy[i] = sf[(4 * N + i) * S];
    }
    if (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N; i += 4) {
            const int4 a = *reinterpret_cast<const int4 *>(actions + env * N + i);
            act[i] = a.x; act[i + 1] = a.y; act[i + 2] = a.z; act[i + 3] = a.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; i++) act[i] = actions[env * N + i];
    }
    const int steps = si[0] + 1;                  // episode_steps += 1: first line of every step()
    const bool prev_valid = si[S] != 0;
    // PredatorCapturePrey: the prey positions are fetched now, with the rest of the state, into a thread-private array;
    // loading them inside the tail's loop over the prey put one global round trip per prey on the critical path
    double prey_xy[SCN == MRB_PCP ? 2 * MRB_MAX_PREY : 1];
    if (SCN == MRB_PCP) {
        for (int q = 0; q < 2 * c.num_prey; q++) prey_xy[q] = scf[q * S];
    }
    int at_pix = 0, at_reached = 0;
    if (SCN == MRB_ARCTIC) { at_pix = sci[7 * S]; at_reached = sci[8 * S]; }

    // roboEnv.py:42 -> _generate_step_goal_positions: goals from the pose at entry
    double gx[N], gy[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
        const int a = SCN == MRB_MATERIAL ? act[i] / 4 : act[i];           // MaterialTransport.py:23
        generate_goal(c, agent_step_size<SCN, N>(c, i, at_pix), a, px[i], py[i], gx[i], gy[i]);
    }

    // dtv = dt v, dtw = dt omega: the velocities in force, pre-multiplied by the time step
    double dtv[N], dtw[N], cs[N], sn[N], cd[N], sd[N], dist[N];
#pragma unroll
    for (int i = 0; i < N; i++) dist[i] = 0.0;
    if (c.track_dist && prev_valid) {             // roboEnv.py:55-56 at sub-step 0
#pragma unroll
        for (int i = 0; i < N; i++) {
            const double dx = px[i] - qx[i], dy = py[i] - qy[i], n2 = dx * dx + dy * dy;
            dist[i] = n2 > 1e-200 ? n2 * fast_rsqrt(n2) : 0.0;             // |pose - previous pose|
        }
    }
    int msg = 0, n_qp = 0, n_it = 0, n_stall = 0, n_itw = 0;
    const int UF = c.update_frequency;
    const double coff = c.collision_offset;
    auto wrap = [](double t) { return t > kPi ? t - kTwoPi : (t < -kPi ? t + kTwoPi : t); };
    // roboEnv.py:52-96 as two nested loops: a controller evaluation (k % 15 == 0, or every sub-step on the Robotarium,
    // :63-65), then the sub-steps that run with its velocities.  The inner loop is validation + Euler update only.
    int k = 0;
    while (k < UF) {
        {
            double xix[N], xiy[N], ux[N], uy[N];
#pragma unroll
            for (int i = 0; i < N; i++) {
                heading_sincos(th[i], sn[i], cs[i]);
                xix[i] = px[i] + kProjectionDistance * cs[i];              // uni_to_si_states (A.7)
                xiy[i] = py[i] + kProjectionDistance * sn[i];
                double dx = gx[i] - xix[i], dy = gy[i] - xiy[i];           // si_position_controller (A.6)
                const double n2 = dx * dx + dy * dy;
                if (n2 > kSiVelocityLimit * kSiVelocityLimit) {              // |dxi| > 0.15: scale to 0.15 (no sqrt, no division)
                    const double sc = kSiVelocityLimit * fast_rsqrt(n2);
                    dx *= sc; dy *= sc;
                }
                ux[i] = dx; uy[i] = dy;
            }
            // Teams of 5 and 6 robots: the solver alone needs more than the 255 registers (it spills inside its iteration
            // loop even as a stand-alone kernel), and whatever else is live across the call makes that worse - measured
            // 205 local loads + 117 stores per iteration here against 110 + 69 alone.  So everything that is only needed
            // AFTER the solve is parked in local memory by hand (one store and one load per value and controller
            // evaluation); volatile, so that the compiler cannot keep register copies alive across the solve.  Teams of
            // up to 4 robots park too (measured: 0.159 -> 0.154 ms, PCP 65,536 envs).
            volatile double park[8 * N];
            volatile int park_act[N];
#pragma unroll
            for (int i = 0; i < N; i++) {
                park[i] = px[i]; park[N + i] = py[i]; park[2 * N + i] = th[i]; park[3 * N + i] = gx[i];
                park[4 * N + i] = gy[i]; park[5 * N + i] = dist[i]; park[6 * N + i] = cs[i]; park[7 * N + i] = sn[i];
                park_act[i] = act[i];
            }
            const int it = qp_run<N>(xix, xiy, ux, uy, c.barrier_default != 0, qp_smem);    // controller.py:23
#pragma unroll
            for (int i = 0; i < N; i++) {
                px[i] = park[i]; py[i] = park[N + i]; th[i] = park[2 * N + i]; gx[i] = park[3 * N + i];
                gy[i] = park[4 * N + i]; dist[i] = park[5 * N + i]; cs[i] = park[6 * N + i]; sn[i] = park[7 * N + i];
                act[i] = park_act[i];
            }
            n_it += it;
            n_stall += it >= 25;
            n_qp++;
            if (c.collect_stats) {                 // the warp iterated until its slowest env converged
                const unsigned here = __activemask();
                n_itw += __reduce_max_sync(here, it);
            }
#pragma unroll
            for (int i = 0; i < N; i++) {                                   // si_to_uni_dyn (A.7) + saturation (A.2)
                const double vv = cs[i] * ux[i] + sn[i] * uy[i];
                double ww = (1.0 / kProjectionDistance) * (-sn[i] * ux[i] + cs[i] * uy[i]);
                ww = clampd(ww, -kAngularLimit, kAngularLimit);
                dtv[i] = kTimeStep * clampd(vv, -kMaxLinearVelocity, kMaxLinearVelocity);
                dtw[i] = kTimeStep * clampd(ww, -kMaxAngularVelocity, kMaxAngularVelocity);
                small_sincos(dtw[i], sd[i], cd[i]);
            }
        }
        const int left = UF - k;
        const int run = c.robotarium ? 1 : (c.ctrl_period < left ? c.ctrl_period : left);
        int since = 0;                             // updates made with these velocities
        for (int j = 0; j < run; j++) {
            // Robotarium.step (A.3): _validate (A.4) on the entering pose, then Euler update in place
            bool viol_b = false;
#pragma unroll
            for (int i = 0; i < N; i++)
                viol_b |= (px[i] < kArenaXMin) | (px[i] > kArenaXMax) | (py[i] < kArenaYMin) | (py[i] > kArenaYMax);
            // collision points: the centres, or (collision_offset != 0) the points projected along the heading;
            // (cs, sn) is the heading of the entering pose (fresh at the evaluation, advanced with the pose since).
            // A pair collides when thr2 - |d|^2 >= 0, i.e. when the sign bit of that difference is clear: the bits
            // are AND-ed in the integer pipe (one FP64 compare per pair costs more, and the compiler would turn an
            // OR of compares into a chain of NaN-aware fmin)
            double cxp[N], cyp[N];
#pragma unroll
            for (int i = 0; i < N; i++) { cxp[i] = fma(coff, cs[i], px[i]); cyp[i] = fma(coff, sn[i], py[i]); }
            int clear = -1;
#pragma unroll
            for (int i = 0; i < N - 1; i++)
#pragma unroll
                for (int jj = i + 1; jj < N; jj++) {
                    const double dx = cxp[i] - cxp[jj], dy = cyp[i] - cyp[jj];
                    clear &= __double2hiint(fma(-dy, dy, fma(-dx, dx, p.collision_thr2)));
                }
            const bool viol_c = clear >= 0;
#pragma unroll
            for (int i = 0; i < N; i++) {
                px[i] = fma(dtv[i], cs[i], px[i]);
                py[i] = fma(dtv[i], sn[i], py[i]);
                th[i] += dtw[i];
                const double c2 = cs[i] * cd[i] - sn[i] * sd[i];           // heading advanced by dt*omega
                sn[i] = sn[i] * cd[i] + cs[i] * sd[i];
                cs[i] = c2;
            }
            since++;
            if (c.penalize_violations && (viol_c || viol_b)) {              // roboEnv.py:82-94
                msg = (viol_c ? 1 : 0) + (viol_b ? 2 : 0);
                break;
            }
        }
        k += since;
        // roboEnv.py:55-56 adds |pose_k - pose_{k-1}| = dt |v_{k-1}| (c^2 + s^2 = 1) at every sub-step k >= 1, i.e. one
        // sub-step late: the last update of a step that ran to the end is counted by the NEXT step (through the
        // stored previous pose); after a violation roboEnv.py:93 adds it right away
        const double cnt = (double)((msg || k < UF) ? since : since - 1);
#pragma unroll
        for (int i = 0; i < N; i++) {
            dist[i] = fma(cnt, fabs(dtv[i]), dist[i]);
            // the reference wraps the heading with atan2(sin, cos) after every sub-step; |dt omega| <= 0.12, so the sum
            // of up to ctrl_period increments is brought back into (-pi, pi] by one conditional +-2 pi
            th[i] = wrap(th[i]);
        }
        if (msg) break;
    }
    const int n_sub = k;
    // roboEnv.py:59 previous_pose = the pose entering the last sub-step that ran: the final pose stepped back by that
    // update (heading rotated back by dt*omega); agrees with a stored copy to an ulp and costs no registers in the loop
#pragma unroll
    for (int i = 0; i < N; i++) {
        const double cp = cs[i] * cd[i] + sn[i] * sd[i], sp = sn[i] * cd[i] - cs[i] * sd[i];
        qx[i] = fma(-dtv[i], cp, px[i]);
        qy[i] = fma(-dtv[i], sp, py[i]);
    }

    // ---------------------------------------------------------------- scenario tail (order matters)
    const int D = p.obs_dim;
    float *obs = p.buf.obs + env * (int64_t)(N * D);
    double *obs64 = p.buf.obs_f64 ? p.buf.obs_f64 + env * (int64_t)(N * D) : nullptr;
    double *rew64 = p.buf.reward_f64 ? p.buf.reward_f64 + env * N : nullptr;
    float rew[N];
    bool done = false;
    int remaining = 0, scen_metric = 0;

    if (SCN == MRB_PCP) {
        const int P = c.num_prey;
        uint32_t sensed = (uint32_t)sci[0], captured = (uint32_t)sci[S];
        const int unseen0 = P - __popc(sensed), left0 = P - __popc(captured);
        double bd[N], bx[N], by[N];
#pragma unroll
        for (int a = 0; a < N; a++) { bd[a] = -1.0; bx[a] = -5.0; by[a] = -5.0; }
        for (int q = 0; q < P; q++) {
            if ((captured >> q) & 1) continue;
            const double qxp = prey_xy[2 * q], qyp = prey_xy[2 * q + 1];
            double d2[N];
            bool sense = false, capture = false;
#pragma unroll
            for (int a = 0; a < N; a++) {
                const double dx = px[a] - qxp, dy = py[a] - qyp;
                d2[a] = dx * dx + dy * dy;
                // _update_tracking_and_locations (PredatorCapturePrey.py:72-95): predators sense
                // (capture agents have sensing radius 0), capture agents capture on 'no_action'
                const bool pred = a < c.num_predators;
                sense |= d2[a] <= (pred ? p.sense_thr2 : 0.0);
                capture |= (act[a] == 4) && d2[a] <= (pred ? 0.0 : p.capture_thr2);
            }
            if (sense) sensed |= 1u << q;
            if (((sensed >> q) & 1) && capture) { captured |= 1u << q; continue; }
            // Agent.get_observation (agent.py:19-46): closest uncaptured prey inside own sensing radius.  The
            // reference compares the ROUNDED norms (utilities/misc.py:14-18 is_close) with a strict `<`, so two prey
            // whose squared distances differ by an ulp but round to the same norm keep the first one
#pragma unroll
            for (int a = 0; a < N; a++) {
                const bool in_range = d2[a] <= (a < c.num_predators ? p.sense_thr2 : 0.0);
                if (in_range) {
                    const double dd = neighbor_dist(px[a] - qxp, py[a] - qyp);
                    if (bd[a] < 0.0 || dd < bd[a]) { bd[a] = dd; bx[a] = qxp; by[a] = qyp; }
                }
            }
        }
        const int unseen = P - __popc(sensed), left = P - __popc(captured);
        sci[0] = (int32_t)sensed; sci[S] = (int32_t)captured;
        // get_observations (PredatorCapturePrey.py:178-207)
        const int od = c.capability_aware ? 6 : 4;
#pragma unroll
        for (int a = 0; a < N; a++) {
            int slot = 0;
            auto put = [&](int b) {
                const ObsRow o(obs, obs64, a * D + slot * od);
                o.put(0, px[b]); o.put(1, py[b]); o.put(2, bx[b]); o.put(3, by[b]);
                if (od == 6) {
                    o.put(4, b < c.num_predators ? c.predator_radius : 0.0);
                    o.put(5, b < c.num_predators ? 0.0 : c.capture_radius);
                }
                slot++;
            };
            put(a);
            if (c.num_neighbors >= N - 1) {
#pragma unroll
                for (int b = 0; b < N; b++) if (b != a) put(b);
            } else {                                   // utilities/misc.py:20-25: K nearest, ascending distance
                uint32_t used = 1u << a;
                for (int kk = 0; kk < c.num_neighbors; kk++) {
                    int best = -1; double bdist = 0.0;
#pragma unroll
                    for (int b = 0; b < N; b++) {
                        const double dx = px[b] - px[a], dy = py[b] - py[a], dd = neighbor_dist(dx, dy);
                        if (!((used >> b) & 1) && (best < 0 || dd < bdist)) { best = b; bdist = dd; }
                    }
                    used |= 1u << best;
#pragma unroll
                    for (int b = 0; b < N; b++) if (b == best) put(b);
                }
            }
        }
        double r;
        if (msg) { r = c.violation_reward; done = true; }                  // PredatorCapturePrey.py:155-159
        else {                                                             // get_rewards (:209-216)
            r = ((unseen0 - unseen) * c.sense_reward + (left0 - left) * c.capture_reward) + c.time_penalty;
            done = steps > c.max_episode_steps || left == 0;
        }
#pragma unroll
        for (int a = 0; a < N; a++) { rew[a] = (float)r; if (rew64) rew64[a] = r; }
        remaining = left; scen_metric = P - left;
    } else if (SCN == MRB_WAREHOUSE) {
        uint32_t loaded = (uint32_t)sci[0];
#pragma unroll
        for (int a = 0; a < N; a++) {                                       // get_observations (warehouse.py:124-143)
            int slot = 0;
            auto put = [&](int b) {
                const ObsRow o(obs, obs64, a * D + slot * 3);
                o.put(0, px[b]); o.put(1, py[b]); o.put(2, (double)((loaded >> b) & 1));
                slot++;
            };
            put(a);
            if (c.num_neighbors >= N - 1) {
#pragma unroll
                for (int b = 0; b < N; b++) if (b != a) put(b);
            } else {
                uint32_t used = 1u << a;
                for (int kk = 0; kk < c.num_neighbors; kk++) {
                    int best = -1; double bdist = 0.0;
#pragma unroll
                    for (int b = 0; b < N; b++) {
                        const double dx = px[b] - px[a], dy = py[b] - py[a], dd = neighbor_dist(dx, dy);
                        if (!((used >> b) & 1) && (best < 0 || dd < bdist)) { best = b; bdist = dd; }
                    }
                    used |= 1u << best;
#pragma unroll
                    for (int b = 0; b < N; b++) if (b == best) put(b);
                }
            }
        }
        if (msg) {
#pragma unroll
            for (int a = 0; a < N; a++) { rew[a] = (float)c.violation_reward; if (rew64) rew64[a] = c.violation_reward; }
            done = true;
        } else {                                                            // get_rewards (:145-178)
#pragma unroll
            for (int a = 0; a < N; a++) {
                const bool green = (a % 2 == 0), ld = (loaded >> a) & 1;    // even index -> Green (:63-65)
                double r = 0.0;
                if (ld) {
                    if (px[a] < -1.5 + c.goal_width && ((green && py[a] > 0) || (!green && py[a] <= 0))) {
                        r = c.unload_reward; loaded &= ~(1u << a); scen_metric++;
                    }
                } else {
                    if (px[a] > 1.5 - c.goal_width && ((!green && py[a] > 0) || (green && py[a] <= 0))) {
                        r = c.load_reward; loaded |= 1u << a;
                    }
                }
                rew[a] = (float)r;
                if (rew64) rew64[a] = r;
            }
            done = steps > c.max_episode_steps;
        }
        sci[0] = (int32_t)loaded;
    } else if (SCN == MRB_MATERIAL) {
        int load[N], zone[2];
#pragma unroll
        for (int a = 0; a < N; a++) load[a] = sci[a * S];
        zone[0] = sci[N * S]; zone[1] = sci[(N + 1) * S];
        int messages = 0;
#pragma unroll
        for (int i = 0; i < 4 && i < N; i++) messages |= (act[i] % 4) << (2 * i);   // MaterialTransport.py:119-120
#pragma unroll
        for (int a = 0; a < N; a++) {                                       // get_observations (:150-159)
            const ObsRow o(obs, obs64, a * D);
            o.put(0, px[a]); o.put(1, py[a]); o.put(2, (double)load[a]);
            o.put(3, (double)zone[0]); o.put(4, (double)zone[1]);
#pragma unroll
            for (int i = 0; i < 4; i++) o.put(5 + i, (double)((messages >> (2 * i)) & 3));
            if (c.capability_aware) {
                o.put(9, (double)(a < c.n_fast ? c.small_torque : c.large_torque));
                o.put(10, a < c.n_fast ? c.fast_step : c.slow_step);
            }
        }
        double r;
        if (msg) { r = c.violation_reward; done = true; }
        else {                                                              // get_reward (:161-189)
            r = c.time_penalty;
#pragma unroll
            for (int a = 0; a < N; a++) {
                const int torque = a < c.n_fast ? c.small_torque : c.large_torque;
                if (load[a] > 0) {
                    if (px[a] < -1.5 + c.goal_width) { r += load[a] * c.unload_reward; scen_metric += load[a]; load[a] = 0; }
                } else {
                    int zi = -1;
                    if (px[a] > 1.5 - c.goal_width) zi = 1;
                    else if (px[a] * px[a] + py[a] * py[a] <= p.zone1_thr2) zi = 0;
                    if (zi >= 0) {
                        const int zl = zi ? zone[1] : zone[0];
                        const int take = zl > torque ? torque : zl;
                        load[a] = take;
                        if (zi) zone[1] = zl - take; else zone[0] = zl - take;
                        r += take * c.load_reward;
                    }
                }
            }
            done = steps > c.max_episode_steps;
            if (!done) {
                bool empty = zone[0] == 0 && zone[1] == 0;
#pragma unroll
                for (int a = 0; a < N; a++) empty &= load[a] == 0;
                done = empty;
            }
        }
        remaining = zone[0] + zone[1];
#pragma unroll
        for (int a = 0; a < N; a++) { rew[a] = (float)r; if (rew64) rew64[a] = r; remaining += load[a]; sci[a * S] = load[a]; }
        sci[N * S] = zone[0]; sci[(N + 1) * S] = zone[1]; sci[(N + 2) * S] = messages;
    } else if (SCN == MRB_ARCTIC) {
        uint32_t g[6];
#pragma unroll
        for (int t = 0; t < 6; t++) g[t] = (uint32_t)sci[t * S];
        const int goal_col = sci[6 * S];
        int row[N], col[N], pix[N];
#pragma unroll
        for (int i = 0; i < N; i++) {
            arctic_cell(px[i], py[i], row[i], col[i]);
            pix[i] = arctic_grid(g, row[i], col[i]);
        }
        const double goalx = goal_col * .25 - 1.5, goaly = (-1 * .25 + .75);  // get_pose_from_cell([1, g])
        int nb[16];
#pragma unroll
        for (int i = 0; i < 2; i++) {                                       // agent.py:73-85
            const int left = col[i] > 0 ? col[i] - 1 : col[i], right = col[i] < 11 ? col[i] + 1 : col[i];
            const int up = row[i] > 0 ? row[i] - 1 : row[i], down = row[i] < 7 ? row[i] + 1 : row[i];
            nb[8 * i + 0] = arctic_grid(g, up, left);   nb[8 * i + 1] = arctic_grid(g, row[i], left);
            nb[8 * i + 2] = arctic_grid(g, down, left); nb[8 * i + 3] = arctic_grid(g, up, col[i]);
            nb[8 * i + 4] = arctic_grid(g, down, col[i]); nb[8 * i + 5] = arctic_grid(g, up, right);
            nb[8 * i + 6] = arctic_grid(g, row[i], right); nb[8 * i + 7] = arctic_grid(g, down, right);
        }
        at_pix = 0;
#pragma unroll
        for (int a = 0; a < N; a++) {                                       // Agent.get_observation (agent.py:14-87)
            at_pix |= pix[a] << (2 * a);
            if (pix[a] == 3) at_reached |= 1 << a;
            constexpr int perm[4][3] = {{1, 2, 3}, {0, 2, 3}, {3, 0, 1}, {2, 0, 1}};   // agent.py:42-69
            const ObsRow o(obs, obs64, a * D);
            o.put(0, px[a]); o.put(1, py[a]); o.put(2, (double)pix[a]);
#pragma unroll
            for (int t = 0; t < 3; t++) {
                const int b = perm[a & 3][t];
                o.put(3 + 3 * t, px[b]); o.put(4 + 3 * t, py[b]); o.put(5 + 3 * t, (double)pix[b]);
            }
            o.put(12, goalx); o.put(13, goaly);
#pragma unroll
            for (int t = 0; t < 16; t++) o.put(14 + t, (double)nb[t]);
        }
        double r;
        if (msg) { r = c.violation_reward; done = true; }
        else {                                                              // get_reward (ArcticTransport.py:125-134)
            r = 0.0;
            bool all_reached = true;
#pragma unroll
            for (int a = 2; a < N; a++) {
                const bool reached = (at_reached >> a) & 1;
                if (!reached) r += c.not_reached_penalty;
                if (pix[a] != 3) {
                    const double dx = px[a] - goalx, dy = py[a] - goaly;
                    r += c.dist_multiplier * (dx * dx + dy * dy);
                }
                all_reached &= reached;
            }
            done = steps > c.max_episode_steps || all_reached;
            scen_metric = all_reached ? 1 : 0;
        }
#pragma unroll
        for (int a = 0; a < N; a++) { rew[a] = (float)r; if (rew64) rew64[a] = r; }
        sci[7 * S] = at_pix; sci[8 * S] = at_reached;
    } else {                                                                // Simple (simple.py:155-225)
        const double goalx = scf[0], goaly = scf[S];
#pragma unroll
        for (int a = 0; a < N; a++) {
            const ObsRow o(obs, obs64, a * D);
            int k = 0;
            o.put(k++, px[a]); o.put(k++, py[a]);
#pragma unroll
            for (int b = 0; b < N; b++) if (b != a) { o.put(k++, px[b]); o.put(k++, py[b]); }
            o.put(k++, goalx); o.put(k++, goaly);
            const double dx = px[a] - goalx, dy = py[a] - goaly;
            const double r = msg ? c.violation_reward : -(dx * dx + dy * dy) * c.reward_scaler;
            rew[a] = (float)r;
            if (rew64) rew64[a] = r;
        }
        done = msg != 0 || steps > c.max_episode_steps;
    }

    // ---------------------------------------------------------------- write back
    // the two loads of the tail are issued before the stores, so that their latency runs under them
    const double ep_prev = sf[(5 * N) * S];
    const int32_t episode = c.auto_reset ? si[2 * S] : 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        sf[i * S] = px[i]; sf[(N + i) * S] = py[i]; sf[(2 * N + i) * S] = th[i];
        sf[(3 * N + i) * S] = qx[i]; sf[(4 * N + i) * S] = qy[i];
    }
    si[0] = steps;
    si[S] = 1;
    float team = 0.f;
#pragma unroll
    for (int i = 0; i < N; i++) {
        p.buf.reward[env * N + i] = rew[i];
        team += rew[i];
        if (p.buf.dist) p.buf.dist[env * N + i] = (float)dist[i];
    }
    p.buf.done[env] = done ? 1 : 0;
    p.buf.message[env] = (uint8_t)msg;
    p.buf.remaining[env] = remaining;
    if (p.hout.obs || p.hout.reward || p.hout.done || p.hout.message) {
        // host mirrors.  The observations of a warp's envs are one contiguous block of obs[B][N][D]: re-read it
        // warp-wide so that every store instruction sends 512 contiguous bytes over PCIe.  Only mrb_step_host sets
        // hout, and it launches ranges (never a LIST, whose warps' envs are not contiguous)
        const unsigned act = warp_envs;      // not __activemask(): lanes that diverged above must reconverge here
        __syncwarp(act);
        if (p.hout.obs) {
            const int lane = threadIdx.x & 31, first = __ffs(act) - 1;
            const int64_t env0 = __shfl_sync(act, env, first);
            const int64_t words = (int64_t)__popc(act) * N * D;          // floats; N * D * 4 bytes need not be 16-byte sized
            const float *src = p.buf.obs + env0 * (int64_t)(N * D);
            float *dst = p.hout.obs + env0 * (int64_t)(N * D);
            const int rank = __popc(act & ((1u << lane) - 1));
            const int nact = __popc(act);
            if ((((env0 * N * D) | words) & 3) == 0) {
                const float4 *s4 = reinterpret_cast<const float4 *>(src);
                float4 *d4 = reinterpret_cast<float4 *>(dst);
                for (int64_t k = rank; k < words / 4; k += nact) d4[k] = s4[k];
            } else {
                for (int64_t k = rank; k < words; k += nact) dst[k] = src[k];
            }
        }
        if (p.hout.reward) {
#pragma unroll
            for (int i = 0; i < N; i++) p.hout.reward[env * N + i] = rew[i];
        }
        if (p.hout.done) p.hout.done[env] = done ? 1 : 0;
        if (p.hout.message) p.hout.message[env] = (uint8_t)msg;
    }
    const double ep_return = ep_prev + (double)team;
    sf[(5 * N) * S] = ep_return;

    if (c.collect_stats && p.buf.stats) {
        double *st = p.buf.stats;
        const unsigned active = __activemask();
        const int w_it = __reduce_add_sync(active, n_it), w_qp = __reduce_add_sync(active, n_qp);
        const int w_n = __popc(active), w_stall = __reduce_add_sync(active, n_stall);
        const int w_itw = __reduce_add_sync(active, n_itw), w_sub = __reduce_add_sync(active, n_sub);
        if ((threadIdx.x & 31) == __ffs(active) - 1) {
            atomicAdd(st + MRB_STAT_ENV_STEPS, (double)w_n);
            atomicAdd(st + MRB_STAT_QP_SOLVES, (double)w_qp);
            atomicAdd(st + MRB_STAT_QP_ITERS, (double)w_it);
            atomicAdd(st + MRB_STAT_QP_ITERS_WARP, (double)w_itw);
            atomicAdd(st + MRB_STAT_SUBSTEPS, (double)w_sub);
            if (w_stall) atomicAdd(st + MRB_STAT_QP_STALLS, (double)w_stall);
        }
        if (done) {
            atomicAdd(st + MRB_STAT_EPISODES, 1.0);
            atomicAdd(st + MRB_STAT_RETURN, ep_return);
            atomicAdd(st + MRB_STAT_LENGTH, (double)steps);
            if (msg & 1) atomicAdd(st + MRB_STAT_COLLISION, 1.0);
            if (msg & 2) atomicAdd(st + MRB_STAT_BOUNDARY, 1.0);
            if (!msg && steps > c.max_episode_steps) atomicAdd(st + MRB_STAT_TIMEOUTS, 1.0);
            atomicAdd(st + MRB_STAT_SCENARIO, (double)scen_metric);
        }
    }
    if (done && c.auto_reset) reset_env<SCN>(p, env, episode);
}

template <int SCN, int N>
inline cudaError_t launch_thread(const Params &p, const int32_t *actions, cudaStream_t s)
{
    constexpr int tpb = ThreadShape<N>::kThreads;
    const unsigned grid = (unsigned)((p.env_hi - p.env_lo + tpb - 1) / tpb);
    constexpr size_t smem = QpStore<N>::kBytes;
    const auto kernel = p.envs ? step_thread_kernel<SCN, N, true> : step_thread_kernel<SCN, N>;
    if (smem > 48 * 1024) {
        const cudaError_t attr = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (attr != cudaSuccess) return attr;
    }
    kernel<<<grid, tpb, smem, s>>>(p, actions);
    return cudaGetLastError();
}

}  // namespace mrb
