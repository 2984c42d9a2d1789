// One environment per WARP: the general path for teams that do not fit the one-env-per-thread
// kernel (more than 6 robots, up to 32).  Lane i owns robot i (pose, goal, velocity); the pair
// constraints of the barrier QP are distributed round-robin over the lanes (slot k of lane l is
// pair l + 32 k); the 2N x 2N KKT matrix and the small vectors live in a per-warp shared-memory
// workspace.  Same algorithm, constants and reference citations as step_thread.cuh / qp_thread.cuh.
// With a compile-time team size (20 robots, BASELINE config 5) the Newton system is factored and solved by 8 x 8
// tiles on the FP64 tensor cores (QpWarp::factor_tiles / solve); run-time team sizes use 2 x 2 blocks on the FP64 pipe.
#pragma once
#include <cstdlib>

#include "common.cuh"
#include "launchers.h"
#include "step_thread.cuh"     // ObsRow, reset_env, launch_thread

namespace mrb {

constexpr int kWarpsPerBlock = 4;
constexpr int kWarpMinBlocks = 3;      // 168 registers, 12 warps per SM (the per-constraint vectors that used to force 255 registers are recomputed or read back from the workspace)
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = dmax(__shfl_xor_sync(kFull, v, o), v);
    return v;
}
// FP64 tensor-core tile product D = A (8 x 4, row) * B (4 x 8, col) + C (8 x 8) = one DMMA.8x8x4 on sm_100a.  Lane
// (g = lane / 4, t = lane % 4) holds A[g][t], B[t][g] and C[g][2t], C[g][2t + 1].  Measured on the B200
// (scripts/microbench/dmma.cu, profiles/r02_dmma_microbench.txt): 26 cycles latency, one per 16 cycles and scheduler
// (37 TFLOP/s, and DFMAs issued beside it slow it down) -- the flop rate of 8 warp-DFMAs at full lane use -- so it buys
// instruction slots and lane efficiency, not flops.
__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// D = A * B (C = 0: the zero register, no accumulator to clear)
__device__ __forceinline__ void dmma_8x8x4_zero(double &d0, double &d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%4};" : "=d"(d0), "=d"(d1) : "d"(a), "d"(b), "d"(0.0));
}

// Per-warp shared-memory workspace (doubles).  The Cholesky factor is stored as the lower triangle of
// N x N blocks of 2 x 2 (block (i,k), k <= i, at 4 * (i (i + 1) / 2 + k): [xx, xy, yx, yy] = rows 2i, 2i+1 x
// columns 2k, 2k+1), 32-byte aligned so that a block is two 128-bit shared loads.  Per-pair quantities that the robot
// lanes sum over (w = z/s, right-hand sides, z) are kept as SYMMETRIC N x N matrices with an odd row stride: the lane
// of robot i reads row i with constant offsets and no bank conflicts instead of gathering through the pair index
// (1.6x the conflict-free wavefronts and five integer instructions per element before); the pair's owner writes both
// mirror entries.  The pair directions a_ij = 2 (x_i - x_j) are not stored: they are differences of the doubled
// positions (exact), read as broadcast 128-bit loads.
__host__ __device__ constexpr int pair_row_stride(int N) { return N | 1; }
__host__ __device__ constexpr size_t warp_workspace_doubles(int N)
{
    // factor blocks + six n-vectors + two pair matrices (even) + the inverses of the diagonal 8 x 8 tiles of L
    return ((2 * (size_t)N * (N + 1) + 12 * (size_t)N + 2 * (size_t)N * pair_row_stride(N) + 1) & ~(size_t)1) + 64 * (((size_t)N + 3) / 4);
}
// Compile-time team sizes (the tensor-core solver): exact number of pair slots per lane, and as many warps in ONE CTA per SM
// as the workspace (227 KB) and the register file (168 registers at 12 warps) allow
__host__ __device__ constexpr int team_ppl(int N) { return (N * (N - 1) / 2 + 31) / 32; }
// (register file: 168 registers at 12 warps; small teams need fewer -- measured, 65,536 envs: 8 robots 6.54 ms at 12 warps,
// 5.91 at 16, 5.78 at 20; 12 robots 11.30 / 10.99 / 10.99; 16 robots 17.85 / 17.21 / 18.18)
__host__ __device__ constexpr int team_warps(int N)
{
    const int fit = (int)((227 * 1024) / (warp_workspace_doubles(N) * sizeof(double)));
    const int cap = N <= 8 ? 20 : N <= 16 ? 16 : 12;
    return fit < cap ? fit : cap;
}

// NC: compile-time size of the Newton system in robots, a multiple of 4 (0 = run-time team size, 2 x 2-block code).  The
// tensor-core paths (DMMA tile updates of the factor, tile solves) need it at compile time: their tile loops and predicates
// fold away; with run-time tile counts the same code spills and is slower than the 2 x 2-block code (measured, 20 robots:
// 39.7 vs 28.5 ms).  EXACT: the team has exactly NC robots (loops over robots fold too); otherwise N <= NC robots at run
// time and robots N .. NC - 1 are phantoms without constraints: their rows of K are 2I, their entries of every vector 0.
template <int PPL, int NC = 0, bool EXACT = true>
struct QpWarp {
    static constexpr bool kTiles = NC != 0;
    int N, n, m, lane;
    int NP;                                               // robots the workspace is laid out for (NC, or N)
    int NS;                                               // row stride of the pair matrices
    double *Lb, *invd, *vx, *vq, *vrx, *vdx, *xi2, *Wm, *Ym, *Li;
    int pi[PPL], pj[PPL];
    bool pv[PPL];
    double h[PPL];

    __device__ QpWarp(int N_, double *ws, int lane_) : N(N_), n(2 * N_), m(N_ * (N_ - 1) / 2), lane(lane_)
    {
        NP = kTiles ? NC : N;
        const int np = 2 * NP;
        Lb = ws; invd = Lb + 2 * (size_t)NP * (NP + 1); vx = invd + np; vq = vx + np; vrx = vq + np; vdx = vrx + np;
        NS = pair_row_stride(NP);
        xi2 = vdx + np;                                   // (2 x_i, 2 y_i), interleaved
        Wm = xi2 + np; Ym = Wm + (size_t)NP * NS;         // Ym holds z or the right-hand-side multipliers (never live together)
        Li = ws + (warp_workspace_doubles(NP) - 64 * (((size_t)NP + 3) / 4));    // dense row-major 8 x 8 per diagonal tile
        if (kTiles && !EXACT) {                           // phantom robots: no weights, zero vectors (never written afterwards)
            for (int k = lane; k < 2 * NP * NS; k += 32) Wm[k] = 0.0;
            for (int k = 2 * N + lane; k < np; k += 32) { vx[k] = 0.0; vq[k] = 0.0; vrx[k] = 0.0; vdx[k] = 0.0; xi2[k] = 0.0; }
            __syncwarp();
        }
#pragma unroll
        for (int k = 0; k < PPL; k++) {                   // decode my pair slots once
            const int c = lane + 32 * k;
            pv[k] = c < m;
            int i = 0, rem = pv[k] ? c : 0;
            while (i < N - 2 && rem >= N - 1 - i) { rem -= N - 1 - i; i++; }     // i <= N - 2: terminates for every N >= 2
            pi[k] = i; pj[k] = i + 1 + rem;
        }
    }
    __device__ __forceinline__ double *blk(int i, int k) const { return Lb + 4 * (size_t)(i * (i + 1) / 2 + k); }

    // (G v)_c for my pair slots; the pair directions a_c are recomputed from the doubled positions (keeping them in
    // registers costs 2 PPL doubles per lane, which is what caps the kernel at 8 warps per SM)
    __device__ __forceinline__ void G_mul(const double *v, double (&out)[PPL]) const
    {
        const double2 *v2 = reinterpret_cast<const double2 *>(v), *x2 = reinterpret_cast<const double2 *>(xi2);
#pragma unroll
        for (int k = 0; k < PPL; k++) {
            const double2 xa = x2[pi[k]], xb = x2[pj[k]], va = v2[pi[k]], vb = v2[pj[k]];
            out[k] = pv[k] ? (xa.x - xb.x) * (vb.x - va.x) + (xa.y - xb.y) * (vb.y - va.y) : 0.0;
        }
    }
    // both mirror entries of a pair matrix
    __device__ __forceinline__ void pair_store(double *M, int k, double v) const { M[pi[k] * NS + pj[k]] = v; M[pj[k] * NS + pi[k]] = v; }
    __device__ __forceinline__ double pair_load(const double *M, int k) const { return M[pi[k] * NS + pj[k]]; }
    // out (smem, robot lanes) += G' y, y a pair matrix: (G'y)_i = -sum_j a_ij y_ij with a_ij = 2 (x_i - x_j) seen from
    // robot i (the diagonal entry of the matrix is 0 and a_ii = 0)
    __device__ __forceinline__ void GT_acc(const double *y, double *out) const
    {
        if (lane < N) {
            const double2 *x2 = reinterpret_cast<const double2 *>(xi2);
            const double2 me2 = x2[lane];
            const double *row = y + lane * NS;
            double sx = 0.0, sy = 0.0, sx1 = 0.0, sy1 = 0.0;        // even / odd terms: half the dependent depth
            int j = 0;
            for (; j + 1 < N; j += 2) {
                const double2 o = x2[j], o1 = x2[j + 1];
                const double t = row[j], t1 = row[j + 1];
                sx = fma(me2.x - o.x, t, sx); sy = fma(me2.y - o.y, t, sy);
                sx1 = fma(me2.x - o1.x, t1, sx1); sy1 = fma(me2.y - o1.y, t1, sy1);
            }
            if (j < N) { const double2 o = x2[j]; const double t = row[j]; sx = fma(me2.x - o.x, t, sx); sy = fma(me2.y - o.y, t, sy); }
            out[2 * lane] -= sx + sx1; out[2 * lane + 1] -= sy + sy1;
        }
    }
    // K := 2I + G' diag(w) G as the lower triangle of 2 x 2 blocks (lane i builds block row i)
    __device__ __forceinline__ void assemble()
    {
        __syncwarp();
        const int NA = kTiles ? NC : N;                     // the tile path also builds the (2I) rows of phantom robots
        if (lane < NA) {
            double dxx = 2.0, dxy = 0.0, dyy = 2.0;
            const double2 *x2 = reinterpret_cast<const double2 *>(xi2);
            const double2 me2 = x2[lane];
            const double *wrow = Wm + lane * NS;
            for (int j = 0; j < NA; j++) {
                const double2 xo = x2[j];
                const double w = wrow[j], a = me2.x - xo.x, b = me2.y - xo.y;    // w_ii = 0
                const double wa = w * a, wb = w * b;
                const double pxx = wa * a, pxy = wa * b, pyy = wb * b;
                dxx += pxx; dxy += pxy; dyy += pyy;
                if (j < lane) {
                    double2 *o = reinterpret_cast<double2 *>(blk(lane, j));
                    o[0] = make_double2(-pxx, -pxy); o[1] = make_double2(-pxy, -pyy);
                }
            }
            double2 *o = reinterpret_cast<double2 *>(blk(lane, lane));
            o[0] = make_double2(dxx, 0.0); o[1] = make_double2(dxy, dyy);
        }
        __syncwarp();
    }
    // K -> its Cholesky factor, in place; invd = reciprocals of the diagonal of L
    __device__ void factor()
    {
        assemble();
        if constexpr (kTiles) { factor_tiles(); return; }
        const bool me = lane < N;
        const double2 *ri = reinterpret_cast<const double2 *>(blk(me ? lane : 0, 0));
        // Left-looking by 2 x 2 blocks, lane i owns block row i.  Diagonal block from S (every lane runs the arithmetic,
        // lane j's result is broadcast and stored), then L_ij = S L_jj^-T for the rows below; returns the new block of
        // this lane in (x00, x01, x10, x11)
        auto finish_column = [&](int j, double sxx, double sxy, double syx, double syy, double &x00, double &x01, double &x10, double &x11) {
            double r1 = fast_rsqrt(sxx);
            double l21 = syx * r1;
            const double d2 = fma(-l21, l21, syy);
            double r2 = fast_rsqrt(d2);
            if (lane == j) {
                double2 *o = reinterpret_cast<double2 *>(blk(j, j));
                o[0] = make_double2(sxx * r1, 0.0); o[1] = make_double2(l21, d2 * r2);
                invd[2 * j] = r1; invd[2 * j + 1] = r2;
            }
            r1 = __shfl_sync(kFull, r1, j); l21 = __shfl_sync(kFull, l21, j); r2 = __shfl_sync(kFull, r2, j);
            x00 = sxx * r1; x10 = syx * r1;
            x01 = fma(-x00, l21, sxy) * r2; x11 = fma(-x10, l21, syy) * r2;
            if (me && lane > j) {
                double2 *o = reinterpret_cast<double2 *>(blk(lane, j));
                o[0] = make_double2(x00, x01); o[1] = make_double2(x10, x11);
            }
        };
        int j = 0;
        // two block columns per sweep: one load of this lane's block (i,k) feeds the updates of S_ij and S_i,j+1
        // (16 FMAs per two lane-varying and four broadcast 128-bit loads instead of 8 per two and two)
        for (; j + 1 < N; j += 2) {
            double axx = 1.0, axy = 0.0, ayx = 0.0, ayy = 1.0, bxx = 1.0, bxy = 0.0, byx = 0.0, byy = 1.0;
            if (me && lane >= j) {
                const double2 *rj = reinterpret_cast<const double2 *>(blk(j, 0));
                const double2 *rj1 = reinterpret_cast<const double2 *>(blk(j + 1, 0));
                const double2 a0 = ri[2 * j], a1 = ri[2 * j + 1];
                axx = a0.x; axy = a0.y; ayx = a1.x; ayy = a1.y;
                if (lane > j) { const double2 b0 = ri[2 * j + 2], b1 = ri[2 * j + 3]; bxx = b0.x; bxy = b0.y; byx = b1.x; byy = b1.y; }
                for (int k = 0; k < j; k++) {
                    const double2 i0 = ri[2 * k], i1 = ri[2 * k + 1], p0 = rj[2 * k], p1 = rj[2 * k + 1], q0 = rj1[2 * k], q1 = rj1[2 * k + 1];
                    axx = fma(-i0.x, p0.x, axx); axx = fma(-i0.y, p0.y, axx);
                    axy = fma(-i0.x, p1.x, axy); axy = fma(-i0.y, p1.y, axy);
                    ayx = fma(-i1.x, p0.x, ayx); ayx = fma(-i1.y, p0.y, ayx);
                    ayy = fma(-i1.x, p1.x, ayy); ayy = fma(-i1.y, p1.y, ayy);
                    bxx = fma(-i0.x, q0.x, bxx); bxx = fma(-i0.y, q0.y, bxx);
                    bxy = fma(-i0.x, q1.x, bxy); bxy = fma(-i0.y, q1.y, bxy);
                    byx = fma(-i1.x, q0.x, byx); byx = fma(-i1.y, q0.y, byx);
                    byy = fma(-i1.x, q1.x, byy); byy = fma(-i1.y, q1.y, byy);
                }
            }
            double x00, x01, x10, x11;
            finish_column(j, axx, axy, ayx, ayy, x00, x01, x10, x11);
            // the k = j term of column j + 1 needs L_(j+1),j, which lane j + 1 has just computed
            const double t00 = __shfl_sync(kFull, x00, j + 1), t01 = __shfl_sync(kFull, x01, j + 1);
            const double t10 = __shfl_sync(kFull, x10, j + 1), t11 = __shfl_sync(kFull, x11, j + 1);
            bxx = fma(-x00, t00, bxx); bxx = fma(-x01, t01, bxx);
            bxy = fma(-x00, t10, bxy); bxy = fma(-x01, t11, bxy);
            byx = fma(-x10, t00, byx); byx = fma(-x11, t01, byx);
            byy = fma(-x10, t10, byy); byy = fma(-x11, t11, byy);
            if (!(me && lane > j)) { bxx = 1.0; bxy = 0.0; byx = 0.0; byy = 1.0; }      // lanes without a row in column j + 1
            double y00, y01, y10, y11;
            finish_column(j + 1, bxx, bxy, byx, byy, y00, y01, y10, y11);
            __syncwarp();
        }
        if (j < N) {                                        // odd team size: the last block column on its own
            double sxx = 1.0, sxy = 0.0, syx = 0.0, syy = 1.0;
            if (me && lane >= j) {
                const double2 *rj = reinterpret_cast<const double2 *>(blk(j, 0));
                const double2 a0 = ri[2 * j], a1 = ri[2 * j + 1];
                sxx = a0.x; sxy = a0.y; syx = a1.x; syy = a1.y;
                for (int k = 0; k < j; k++) {
                    const double2 i0 = ri[2 * k], i1 = ri[2 * k + 1], p0 = rj[2 * k], p1 = rj[2 * k + 1];
                    sxx = fma(-i0.x, p0.x, sxx); sxx = fma(-i0.y, p0.y, sxx);
                    sxy = fma(-i0.x, p1.x, sxy); sxy = fma(-i0.y, p1.y, sxy);
                    syx = fma(-i1.x, p0.x, syx); syx = fma(-i1.y, p0.y, syx);
                    syy = fma(-i1.x, p1.x, syy); syy = fma(-i1.y, p1.y, syy);
                }
            }
            double x00, x01, x10, x11;
            finish_column(j, sxx, sxy, syx, syy, x00, x01, x10, x11);
            __syncwarp();
        }
    }
    // Compile-time team size, a multiple of 4: RIGHT-LOOKING factorisation by pairs of block columns (4 matrix columns)
    // with the trailing updates on the FP64 tensor cores.  Every Schur complement is complete in the workspace when its
    // turn comes, so (1) every lane reads the 4 x 4 diagonal block of the pair with broadcast loads and factors it
    // redundantly -- no shuffles, nothing to wait for from another lane; (2) the lane of every later robot turns its own
    // 2 x 4 strip into L by forward substitution; (3) one DMMA.8x8x4 per trailing 8 x 8 tile subtracts the rank-4
    // contribution of the pair (tiles are read from and written back to the workspace in the accumulator layout).  55
    // DMMAs per factorisation of 20 robots replace 90 left-looking sweeps of 16 DFMAs that ran with 12 to 32 of the 32
    // lanes idle; the inverses of the diagonal 8 x 8 tiles (for solve()) come last.
    __device__ void factor_tiles()
    {
        static_assert(NC % 4 == 0, "the tile path is written for whole 8 x 8 tiles");
        constexpr int TM = NC / 4;
        const bool me = lane < NC;
        double2 *ri = reinterpret_cast<double2 *>(blk(me ? lane : 0, 0));
        const int fg = lane >> 2, ft = lane & 3, fgh = fg >> 1, fa = fg & 1;      // fragment coordinates
        int rowbase[TM];
#pragma unroll
        for (int I = 0; I < TM; I++) { const int i = 4 * I + fgh; rowbase[I] = 2 * i * (i + 1); }
        const int fo = 4 * (ft >> 1) + 2 * fa + (ft & 1);   // A fragment: L[8 I + g][4 jp + t] = Lb[rowbase[I] + 8 jp + fo]
#pragma unroll
        for (int jp = 0; jp < NC / 2; jp++) {               // unrolled: tile ranges, block addresses and most predicates are literals
            const int j = 2 * jp;
            // (1) 4 x 4 diagonal block [[s00], [s10 s11], [s20 s21 s22], [s30 s31 s32 s33]] -> its Cholesky factor
            const double2 *dj = reinterpret_cast<const double2 *>(blk(j, j)), *mj = reinterpret_cast<const double2 *>(blk(j + 1, j)),
                          *ej = reinterpret_cast<const double2 *>(blk(j + 1, j + 1));
            const double2 d0 = dj[0], d1 = dj[1], m0 = mj[0], m1 = mj[1], e0 = ej[0], e1 = ej[1];
            const double r0 = fast_rsqrt(d0.x);
            const double l10 = d1.x * r0, l20 = m0.x * r0, l30 = m1.x * r0;
            const double p1 = fma(-l10, l10, d1.y);
            const double r1 = fast_rsqrt(p1);
            const double l21 = fma(-l20, l10, m0.y) * r1, l31 = fma(-l30, l10, m1.y) * r1;
            const double p2 = fma(-l21, l21, fma(-l20, l20, e0.x));
            const double r2 = fast_rsqrt(p2);
            const double l32 = fma(-l31, l21, fma(-l30, l20, e1.x)) * r2;
            const double p3 = fma(-l32, l32, fma(-l31, l31, fma(-l30, l30, e1.y)));
            const double r3 = fast_rsqrt(p3);
            __syncwarp();                                   // every lane has read the block before it is overwritten
            if (lane == j) {
                double2 *o = reinterpret_cast<double2 *>(blk(j, j));
                o[0] = make_double2(d0.x * r0, 0.0); o[1] = make_double2(l10, p1 * r1);
                *reinterpret_cast<double2 *>(invd + 2 * j) = make_double2(r0, r1);
            } else if (lane == j + 1) {
                double2 *o = reinterpret_cast<double2 *>(blk(j + 1, j));
                o[0] = make_double2(l20, l21); o[1] = make_double2(l30, l31);
                o[2] = make_double2(p2 * r2, 0.0); o[3] = make_double2(l32, p3 * r3);        // block (j + 1, j + 1) follows (j + 1, j)
                *reinterpret_cast<double2 *>(invd + 2 * j + 2) = make_double2(r2, r3);
            } else if (me && lane > j + 1) {
                // (2) rows 2 i, 2 i + 1 of columns 2 j .. 2 j + 3: x L44' = s
                const double2 a0 = ri[2 * j], a1 = ri[2 * j + 1], b0 = ri[2 * j + 2], b1 = ri[2 * j + 3];
                const double x0 = a0.x * r0, y0 = a1.x * r0;
                const double x1 = fma(-x0, l10, a0.y) * r1, y1 = fma(-y0, l10, a1.y) * r1;
                const double x2 = fma(-x1, l21, fma(-x0, l20, b0.x)) * r2, y2 = fma(-y1, l21, fma(-y0, l20, b1.x)) * r2;
                const double x3 = fma(-x2, l32, fma(-x1, l31, fma(-x0, l30, b0.y))) * r3, y3 = fma(-y2, l32, fma(-y1, l31, fma(-y0, l30, b1.y))) * r3;
                ri[2 * j] = make_double2(x0, x1); ri[2 * j + 1] = make_double2(y0, y1);
                ri[2 * j + 2] = make_double2(x2, x3); ri[2 * j + 3] = make_double2(y2, y3);
            }
            __syncwarp();
            if (jp == NC / 2 - 1) break;
            // (3) trailing tiles (I2, J2), J2 >= J0.  After the first pair of a tile column that column is still open:
            // its tiles take part, and only their columns 4 .. 7 (t >= 2) are written back.
            const int J = jp >> 1, half = jp & 1, J0 = J + half;
            double af[TM];
#pragma unroll
            for (int I = 0; I < TM; I++) af[I] = I >= J0 ? Lb[rowbase[I] + 8 * jp + fo] : 0.0;
#pragma unroll
            for (int J2 = 0; J2 < TM; J2++) {
                if (J2 < J0) continue;
                const bool open = J2 == J;                  // (then half == 0)
#pragma unroll
                for (int I2 = 0; I2 < TM; I2++) {
                    if (I2 < J2) continue;
                    const int i = 4 * I2 + fgh, k = 4 * J2 + ft;
                    const bool ok = k <= i && !(open && ft < 2);
                    double2 *cp = reinterpret_cast<double2 *>(Lb + rowbase[I2] + 4 * k + 2 * fa);
                    double2 c = ok ? *cp : make_double2(0.0, 0.0);
                    dmma_8x8x4(c.x, c.y, -af[I2], af[J2]);
                    if (i == k && fa == 0) c.y = 0.0;       // the element above the diagonal of a diagonal block stays 0
                    if (ok) *cp = c;
                }
            }
            __syncwarp();
        }
        // Inverses of the diagonal 8 x 8 tiles of L (the triangular solves multiply by them instead of running four
        // dependent 2 x 2 steps per tile): lane (T, c) = (lane / 8, lane % 8) solves L_TT x = e_c by forward
        // substitution; four tiles per round.
        for (int T0 = 0; T0 < TM; T0 += 4) {
            const int T = T0 + (lane >> 3), c = lane & 7;
            const bool okT = T < TM;
            const int Tc = okT ? T : 0;
            double x[8];
#pragma unroll
            for (int r = 0; r < 8; r++) {
                const int i = 4 * Tc + (r >> 1);
                // row r of the tile: (L[r][2q], L[r][2q + 1]) = blk(i, 4T + q)[2 (r % 2) ..]
                const double2 *row = reinterpret_cast<const double2 *>(Lb + 2 * i * (i + 1) + 16 * Tc + 2 * (r & 1));
                double sum = r == c ? 1.0 : 0.0;
#pragma unroll
                for (int q = 0; 2 * q < r; q++) {
                    const double2 l = row[2 * q];
                    sum = fma(-l.x, x[2 * q], sum);
                    if (2 * q + 1 < r) sum = fma(-l.y, x[2 * q + 1], sum);
                }
                x[r] = sum * invd[8 * Tc + r];
            }
            if (okT) {
#pragma unroll
                for (int r = 0; r < 8; r++) Li[64 * T + 8 * r + c] = x[r];
            }
        }
        __syncwarp();
    }
    // b (smem) := K^-1 b by 8 x 8 tiles on the FP64 tensor cores.  The vector lives in "row layout": lane (g, t) holds
    // element 8 I + g of every tile I (the four lanes of a group hold copies), which is what a DMMA with the vector
    // replicated over the eight columns of B returns in both accumulators.  Forward: y_I = inv(L_II) (b_I - sum_J<I
    // L_IJ y_J); backward: x_I = inv(L_II)' (y_I - sum_J>I L_JI' x_J): five dependent tile steps each way for 20
    // robots instead of twenty 2 x 2 steps with two shuffle broadcasts each.
    __device__ void solve(double *b) const
    {
        if constexpr (kTiles) solve_tiles(b);
        else solve_rows(b);
    }
    __device__ void solve_tiles(double *b) const
    {
        __syncwarp();
        constexpr int TM = NC / 4;                           // whole tiles (static_assert in factor_tiles)
        const int fg = lane >> 2, ft = lane & 3, fgh = fg >> 1, fa = fg & 1;
        const int s0 = 4 * ft, s1 = 16 + 4 * ft;            // lanes holding elements t and 4 + t of a tile in row layout
        double acc[TM > 0 ? TM : 1][2];                     // both accumulators of a tile's DMMAs (equal by construction)
        int rowbase[TM > 0 ? TM : 1];
#pragma unroll
        for (int I = 0; I < TM; I++) {
            const int i = 4 * I + fgh;
            rowbase[I] = 2 * i * (i + 1);
            acc[I][0] = acc[I][1] = b[8 * I + fg];
        }
        // B fragments of a vector held in row layout: lane (g, t) needs elements 4 c + t, c = 0, 1
        auto spread = [&](double v, double &b0, double &b1) { b0 = __shfl_sync(kFull, v, s0); b1 = __shfl_sync(kFull, v, s1); };
        // "Push" order: as soon as a tile of the solution is known it is applied to every later tile, so the DMMAs
        // of one step are independent of each other and only two of them sit between consecutive diagonal steps.
        // The two half products of a diagonal step run in parallel and are added.
#pragma unroll
        for (int J = 0; J < TM; J++) {
            double t0, t1, d0, d1, e0, e1, n0, n1;
            spread(acc[J][0], t0, t1);
            const double *inv = Li + 64 * J + 8 * fg + ft;
            dmma_8x8x4_zero(d0, d1, inv[0], t0);
            dmma_8x8x4_zero(e0, e1, inv[4], t1);
            d0 += e0;
            acc[J][0] = d0;
            spread(-d0, n0, n1);
#pragma unroll
            for (int I = J + 1; I < TM; I++) {
                // L[8 I + g][8 J + 4 c + t]
                const double *src = Lb + rowbase[I] + 16 * J + 4 * (ft >> 1) + 2 * fa + (ft & 1);
                dmma_8x8x4(acc[I][0], acc[I][1], src[0], n0);
                dmma_8x8x4(acc[I][0], acc[I][1], src[8], n1);
            }
        }
#pragma unroll
        for (int I = 0; I < TM; I++) acc[I][1] = acc[I][0];
#pragma unroll
        for (int J = TM - 1; J >= 0; J--) {
            double t0, t1, d0, d1, e0, e1, n0, n1;
            spread(acc[J][0], t0, t1);
            const double *inv = Li + 64 * J + 8 * ft + fg;      // inv(L_JJ)'[g][4 c + t] = inv[4 c + t][g]
            dmma_8x8x4_zero(d0, d1, inv[0], t0);
            dmma_8x8x4_zero(e0, e1, inv[32], t1);
            d0 += e0;
            acc[J][0] = d0;
            spread(-d0, n0, n1);
            // (L_JI)'[g][4 c + t] = L[8 J + 4 c + t][8 I + g], rows 8 J .. of L applied to the earlier tiles I < J
            const int i0 = 4 * J + (ft >> 1), i1 = i0 + 2;
            const double *r0 = Lb + 2 * i0 * (i0 + 1) + 4 * fgh + 2 * (ft & 1) + fa, *r1 = Lb + 2 * i1 * (i1 + 1) + 4 * fgh + 2 * (ft & 1) + fa;
#pragma unroll
            for (int I = J - 1; I >= 0; I--) {
                dmma_8x8x4(acc[I][0], acc[I][1], r0[16 * I], n0);
                dmma_8x8x4(acc[I][0], acc[I][1], r1[16 * I], n1);
            }
        }
        __syncwarp();                                       // the four lanes of a group all read b[8 I + g] above
        if (ft == 0) {
#pragma unroll
            for (int I = 0; I < TM; I++) b[8 * I + fg] = acc[I][0];
        }
        __syncwarp();
    }
    // the same by 2 x 2 blocks: lane i carries (b_2i, b_2i+1), N dependent steps each way (run-time team sizes)
    __device__ void solve_rows(double *b) const
    {
        __syncwarp();
        const bool me = lane < N;
        const int li = me ? lane : 0;
        const double2 *ri = reinterpret_cast<const double2 *>(blk(li, 0));
        double bx = me ? b[2 * li] : 0.0, by = me ? b[2 * li + 1] : 0.0;
        const double r1 = invd[2 * li], r2 = invd[2 * li + 1], l21 = blk(li, li)[2];
        for (int j = 0; j < N; j++) {
            double y0 = bx * r1;
            double y1 = fma(-l21, y0, by) * r2;
            if (lane == j) { bx = y0; by = y1; }
            y0 = __shfl_sync(kFull, y0, j); y1 = __shfl_sync(kFull, y1, j);
            if (me && lane > j) {
                const double2 a0 = ri[2 * j], a1 = ri[2 * j + 1];
                bx = fma(-a0.x, y0, fma(-a0.y, y1, bx));
                by = fma(-a1.x, y0, fma(-a1.y, y1, by));
            }
        }
        for (int i = N - 1; i >= 0; i--) {
            double x1 = by * r2;
            double x0 = fma(-l21, x1, bx) * r1;
            if (lane == i) { bx = x0; by = x1; }
            x0 = __shfl_sync(kFull, x0, i); x1 = __shfl_sync(kFull, x1, i);
            if (lane < i) {                                 // column `lane` of block row i: (L_i,lane)' x_i
                const double2 *rw = reinterpret_cast<const double2 *>(blk(i, lane));
                const double2 a0 = rw[0], a1 = rw[1];
                bx = fma(-a0.x, x0, fma(-a1.x, x1, bx));
                by = fma(-a0.y, x0, fma(-a1.y, x1, by));
            }
        }
        if (me) { b[2 * lane] = bx; b[2 * lane + 1] = by; }
        __syncwarp();
    }

    // lane i < N holds (xi, nominal dxi -> certified u) of robot i.  Returns IPM iterations.
    __device__ int run(double xi_x, double xi_y, double &ux, double &uy, bool barrier_default)
    {
        if (lane < N) {
            const double n2 = ux * ux + uy * uy;
            if (n2 > kQpMagnitudeLimit * kQpMagnitudeLimit) { const double sc = kQpMagnitudeLimit / sqrt(n2); ux *= sc; uy *= sc; }
        }
        if (m == 0) return 0;
        __syncwarp();
        if (lane < N) {
            xi2[2 * lane] = 2.0 * xi_x; xi2[2 * lane + 1] = 2.0 * xi_y;
            Wm[lane * NS + lane] = 0.0; Ym[lane * NS + lane] = 0.0;
            vq[2 * lane] = -2.0 * ux; vq[2 * lane + 1] = -2.0 * uy;
        }
        __syncwarp();
        const double r2 = barrier_default ? 0.17 * 0.17 : 0.2 * 0.2;
        double hh = 0.0;
#pragma unroll
        for (int k = 0; k < PPL; k++) {
            h[k] = 0.0;
            if (pv[k]) {
                const double ex = 0.5 * (xi2[2 * pi[k]] - xi2[2 * pj[k]]), ey = 0.5 * (xi2[2 * pi[k] + 1] - xi2[2 * pj[k] + 1]);
                const double hv = (ex * ex + ey * ey) - r2;
                const double gain = barrier_default ? 100.0 : (hv >= 0.0 ? 100.0 : 1e6);
                h[k] = gain * (hv * hv * hv);
                pair_store(Wm, k, 1.0); pair_store(Ym, k, h[k]);
                hh = fma(h[k], h[k], hh);
            }
        }
        const double qq = warp_sum(lane < N ? 4.0 * (ux * ux + uy * uy) : 0.0);
        hh = warp_sum(hh);
        // (feastol * max(1, |q|))^2 and (feastol * max(1, |h|))^2: cvxopt's residual tests without sqrt / division
        const double feas_x2 = 1e-4 * dmax(qq, 1.0), feas_z2 = 1e-4 * dmax(hh, 1.0);

        // ---- default starting point
        factor();
        if (lane < N) { vx[2 * lane] = -vq[2 * lane]; vx[2 * lane + 1] = -vq[2 * lane + 1]; }
        __syncwarp();
        GT_acc(Ym, vx);
        solve(vx);
        double s[PPL], z[PPL];
        G_mul(vx, z);
        double ss = 0.0, ts = -INFINITY, tz = -INFINITY;
#pragma unroll
        for (int k = 0; k < PPL; k++)
            if (pv[k]) {
                z[k] -= h[k];
                s[k] = -z[k];
                ss = fma(z[k], z[k], ss);
                ts = dmax(z[k], ts);
                tz = dmax(-z[k], tz);
            } else { s[k] = 1.0; z[k] = 1.0; }
        ss = warp_sum(ss); ts = warp_max(ts); tz = warp_max(tz);
        const double nrm = ss > 1.0 ? ss * fast_rsqrt(ss) : 1.0;          // max(|z|, 1)
        double gap = 0.0;
#pragma unroll
        for (int k = 0; k < PPL; k++)
            if (pv[k]) {
                if (ts >= -1e-8 * nrm) s[k] += 1.0 + ts;
                if (tz >= -1e-8 * nrm) z[k] += 1.0 + tz;
                gap = fma(s[k], z[k], gap);
            }
        gap = warp_sum(gap);

        int iters = 0;
        for (; iters <= 50; iters++) {
            // rx = 2x + q + G'z ; rz = s + Gx - h
            double xq = 0.0, xrx = 0.0;
            __syncwarp();
#pragma unroll
            for (int k = 0; k < PPL; k++) if (pv[k]) pair_store(Ym, k, z[k]);
            if (lane < N) {
#pragma unroll
                for (int t = 0; t < 2; t++) {
                    const double xv = vx[2 * lane + t], qv = vq[2 * lane + t], r = fma(2.0, xv, qv);
                    vrx[2 * lane + t] = r;
                    xrx = fma(xv, r, xrx); xq = fma(xv, qv, xq);
                }
            }
            __syncwarp();
            GT_acc(Ym, vrx);
            double rz[PPL];
            G_mul(vx, rz);
            double resx = 0.0, resz = 0.0, zrz = 0.0;
            if (lane < N) resx = vrx[2 * lane] * vrx[2 * lane] + vrx[2 * lane + 1] * vrx[2 * lane + 1];
#pragma unroll
            for (int k = 0; k < PPL; k++)
                if (pv[k]) {
                    rz[k] += s[k] - h[k];
                    resz = fma(rz[k], rz[k], resz);
                    zrz = fma(z[k], rz[k], zrz);
                }
            xq = warp_sum(xq); xrx = warp_sum(xrx); resx = warp_sum(resx); resz = warp_sum(resz); zrz = warp_sum(zrz);
            const double f0 = 0.5 * (xrx + xq);
            const double pcost = f0, dcost = f0 + zrz - gap;
            bool gap_ok = gap <= 1e-7;
            if (pcost < 0.0) gap_ok = gap_ok || (gap <= -1e-2 * pcost);
            else if (dcost > 0.0) gap_ok = gap_ok || (gap <= 1e-2 * dcost);
            if ((resz <= feas_z2 && resx <= feas_x2 && gap_ok) || iters == 50) break;

            // 1/s and 1/z are recomputed where they are used (same function of the same input: identical bits),
            // w = z/s is read back from the workspace and the corrector's (ds, dz) are recomputed in the update
            // pass: 6 PPL fewer live doubles per lane than storing them
            double t2[PPL], gv[PPL];
            __syncwarp();                                   // every lane is done reading z from Ym
#pragma unroll
            for (int k = 0; k < PPL; k++)
                if (pv[k]) {
                    const double w = z[k] * fast_rcp1(s[k]);
                    pair_store(Wm, k, w);
                    pair_store(Ym, k, z[k] - w * rz[k]);
                }
            factor();
            // predictor
            if (lane < N) { vdx[2 * lane] = -vrx[2 * lane]; vdx[2 * lane + 1] = -vrx[2 * lane + 1]; }
            __syncwarp();
            GT_acc(Ym, vdx);
            solve(vdx);
            G_mul(vdx, gv);
            double dsdz = 0.0, tmax = 0.0;
#pragma unroll
            for (int k = 0; k < PPL; k++)
                if (pv[k]) {
                    const double ds = -rz[k] - gv[k];
                    const double dz = -z[k] - pair_load(Wm, k) * ds;
                    t2[k] = ds * dz;
                    dsdz += t2[k];
                    tmax = dmax(dmax(-ds * fast_rcp1(s[k]), -dz * fast_rcp1(z[k])), tmax);
                } else t2[k] = 0.0;
            dsdz = warp_sum(dsdz); tmax = warp_max(tmax);
            double step = tmax <= 1.0 ? 1.0 : fast_rcp(tmax);            // t == 0 ? 1 : min(1, 1/t)
            const double sg = dmin(dmax(1.0 - step + dsdz * fast_rcp(gap) * (step * step), 0.0), 1.0);
            const double sigmamu = sg * sg * sg * (gap / m);
            // corrector
            __syncwarp();
#pragma unroll
            for (int k = 0; k < PPL; k++)
                if (pv[k]) {
                    t2[k] = (sigmamu - t2[k]) * fast_rcp1(s[k]);
                    pair_store(Ym, k, z[k] - pair_load(Wm, k) * rz[k] - t2[k]);
                }
            if (lane < N) { vdx[2 * lane] = -vrx[2 * lane]; vdx[2 * lane + 1] = -vrx[2 * lane + 1]; }
            __syncwarp();
            GT_acc(Ym, vdx);
            solve(vdx);
            G_mul(vdx, gv);
            tmax = 0.0;
#pragma unroll
            for (int k = 0; k < PPL; k++)
                if (pv[k]) {
                    const double ds = -rz[k] - gv[k];
                    const double dz = fma(-pair_load(Wm, k), ds, t2[k] - z[k]);
                    tmax = dmax(dmax(-ds * fast_rcp1(s[k]), -dz * fast_rcp1(z[k])), tmax);
                }
            tmax = warp_max(tmax);
            step = tmax <= 0.99 ? 1.0 : 0.99 * fast_rcp(tmax);           // t == 0 ? 1 : min(1, 0.99/t)
            if (lane < N) { vx[2 * lane] += step * vdx[2 * lane]; vx[2 * lane + 1] += step * vdx[2 * lane + 1]; }
            gap = 0.0;
#pragma unroll
            for (int k = 0; k < PPL; k++)
                if (pv[k]) {
                    const double ds = -rz[k] - gv[k];
                    const double dz = fma(-pair_load(Wm, k), ds, t2[k] - z[k]);
                    s[k] = fma(step, ds, s[k]);
                    z[k] = fma(step, dz, z[k]);
                    gap = fma(s[k], z[k], gap);
                }
            gap = warp_sum(gap);
            __syncwarp();
        }
        if (lane < N) { ux = vx[2 * lane]; uy = vx[2 * lane + 1]; }
        __syncwarp();
        return iters;
    }
};

// ---- the step, lane = robot
// NC: compile-time team size (0 = read it from the config).  With a literal N the pair-index arithmetic, the
// per-robot loops and the block-Cholesky trip counts fold into constants; instantiated for the 20-robot stress
// configuration (BASELINE config 5), every other size takes the generic path.
// WPB: warps (= envs) per CTA.  The 20-robot instantiation runs its 12 resident warps as ONE CTA: they then execute the
// 14 k-instruction body roughly in step and share the instruction fetches (21.8 vs 22.5 ms per 32,768 envs); the generic
// path keeps 4-warp CTAs because the workspace of a 32-robot team would not fit twelve times.
// LIST = {true} (mrb_step_masked): warp i steps env p.envs[i] if i < *p.count, as in step_thread_kernel.
template <int SCN, int PPL, int NC = 0, int WPB = kWarpsPerBlock, bool EXACT = true, bool... LIST>
__global__ void __launch_bounds__(WPB * 32, NC == 0 ? kWarpMinBlocks : 1)
step_warp_kernel(const __grid_constant__ Params p, const int32_t *__restrict__ actions)
{
    constexpr bool kList = (false || ... || LIST);
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t item = (int64_t)blockIdx.x * WPB + wib;
    const int64_t env = kList ? (item < *p.count ? (int64_t)p.envs[item] : -1) : p.env_lo + item;
    if (kList ? env < 0 : env >= p.env_hi) return;
    const mrb_config &c = p.cfg;
    const int N = (NC && EXACT) ? NC : c.num_robots;
    const int64_t S = p.B;
    double *sf = p.buf.state_f64 + env;
    int32_t *si = p.buf.state_i32 + env;
    int32_t *sci = si + kCommonRowsI32 * S;
    double *scf = sf + (5 * N + 1) * S;
    QpWarp<PPL, NC, EXACT> qp(N, smem + (size_t)wib * warp_workspace_doubles(NC ? NC : N), lane);
    const bool me = lane < N;

    double px = 0, py = 0, th = 0, qx = 0, qy = 0;
    int act = 4;
    if (me) {
        px = sf[lane * S]; py = sf[(N + lane) * S]; th = sf[(2 * N + lane) * S];
        qx = sf[(3 * N + lane) * S]; qy = sf[(4 * N + lane) * S];
        act = actions[env * N + lane];
    }
    const int steps = si[0] + 1;
    const bool prev_valid = si[S] != 0;

    double gx = px, gy = py;
    if (me) {
        const int a = SCN == MRB_MATERIAL ? act / 4 : act;
        const double stp = SCN == MRB_MATERIAL ? (lane < c.n_fast ? c.fast_step : c.slow_step) : c.step_dist;
        const double cx = clampd(px, c.left, c.right), cy = clampd(py, c.up, c.down);
        gx = cx; gy = cy;
        if (a == 0) gx = fmax(px - stp, c.left);
        else if (a == 1) gx = fmin(px + stp, c.right);
        else if (a == 2) gy = fmax(py - stp, c.up);
        else if (a == 3) gy = fmin(py + stp, c.down);
    }
    double v = 0, om = 0, cs = 1, sn = 0, cd = 1, sd = 0, dist = 0;
    if (c.track_dist && prev_valid && me) { const double dx = px - qx, dy = py - qy, n2 = dx * dx + dy * dy; dist = n2 > 1e-200 ? n2 * fast_rsqrt(n2) : 0.0; }
    int msg = 0, n_qp = 0, n_it = 0, n_stall = 0, n_sub = 0;
    const int UF = c.update_frequency;
    const double coff = c.collision_offset;
    for (int k = 0; k < UF; k++) {
        n_sub++;
        if (k > 0) dist += kTimeStep * fabs(v);
        qx = px; qy = py;
        if (k % c.ctrl_period == 0 || c.robotarium) {
            double xi_x = 0, xi_y = 0, ux = 0, uy = 0;
            if (me) {
                heading_sincos(th, sn, cs);
                xi_x = px + kProjectionDistance * cs; xi_y = py + kProjectionDistance * sn;
                double dx = gx - xi_x, dy = gy - xi_y;
                const double n2 = dx * dx + dy * dy;
                if (n2 > kSiVelocityLimit * kSiVelocityLimit) { const double sc = kSiVelocityLimit * fast_rsqrt(n2); dx *= sc; dy *= sc; }
                ux = dx; uy = dy;
            }
            const int it = qp.run(xi_x, xi_y, ux, uy, c.barrier_default != 0);
            n_it += it; n_stall += it >= 25; n_qp++;
            if (me) {
                const double vv = cs * ux + sn * uy;
                double ww = (1.0 / kProjectionDistance) * (-sn * ux + cs * uy);
                ww = clampd(ww, -kAngularLimit, kAngularLimit);
                v = clampd(vv, -kMaxLinearVelocity, kMaxLinearVelocity);
                om = clampd(ww, -kMaxAngularVelocity, kMaxAngularVelocity);
                small_sincos(kTimeStep * om, sd, cd);
            }
        }
        bool viol = me && ((px < kArenaXMin) | (px > kArenaXMax) | (py < kArenaYMin) | (py > kArenaYMax));
        const bool viol_b = __any_sync(kFull, viol);
        bool vc = false;
        // collision points: the centres, or (collision_offset != 0) the points projected along the heading
        const double cxp = fma(coff, cs, px), cyp = fma(coff, sn, py);
#pragma unroll
        for (int t = 0; t < PPL; t++) {
            const double xi_ = __shfl_sync(kFull, cxp, qp.pi[t]), yi_ = __shfl_sync(kFull, cyp, qp.pi[t]);
            const double xj_ = __shfl_sync(kFull, cxp, qp.pj[t]), yj_ = __shfl_sync(kFull, cyp, qp.pj[t]);
            const double dx = xi_ - xj_, dy = yi_ - yj_;
            vc |= qp.pv[t] && (dx * dx + dy * dy) <= p.collision_thr2;
        }
        const bool viol_c = __any_sync(kFull, vc);
        if (me) {
            px = px + kTimeStep * cs * v;
            py = py + kTimeStep * sn * v;
            double t = th + kTimeStep * om;
            th = t > kPi ? t - kTwoPi : (t < -kPi ? t + kTwoPi : t);
            const double c2 = cs * cd - sn * sd;
            sn = sn * cd + cs * sd;
            cs = c2;
        }
        if (c.penalize_violations && (viol_c || viol_b)) {
            msg = (viol_c ? 1 : 0) + (viol_b ? 2 : 0);
            dist += kTimeStep * fabs(v);
            break;
        }
    }

    // ---------------------------------------------------------------- scenario tail
    const int D = p.obs_dim;
    const int64_t obs_off = env * (int64_t)(N * D) + (int64_t)lane * D;
    float *obs = p.buf.obs + obs_off;
    double *obs64 = p.buf.obs_f64 ? p.buf.obs_f64 + obs_off : nullptr;
    double rew = 0.0;
    bool done = false;
    int remaining = 0, scen_metric = 0;

    // stage every robot's position in the (now idle) QP workspace so that any lane can read any
    // robot without shuffles inside lane-dependent control flow
    double *spx = qp.xi2, *spy = qp.xi2 + N, *sbx = qp.vx, *sby = qp.vq;
    __syncwarp();
    if (me) { spx[lane] = px; spy[lane] = py; }
    __syncwarp();
    // neighbour order shared by PCP / Warehouse: all others by index, or the K nearest (misc.py:20-25)
    auto for_each_block = [&](auto put) {
        put(lane);
        if (c.num_neighbors >= N - 1) {
            for (int b = 0; b < N; b++) if (b != lane) put(b);
        } else {
            // the rounded norms once (row `lane` of an idle pair matrix), then one compare-and-select pass per neighbour
            double *drow = qp.Wm + lane * qp.NS;
            for (int b = 0; b < N; b++) {
                const double dx = spx[b] - px, dy = spy[b] - py;
                drow[b] = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
            }
            uint32_t used = 1u << lane;
            for (int kk = 0; kk < c.num_neighbors; kk++) {
                int best = -1; double bdist = 0.0;
                for (int b = 0; b < N; b++) {
                    const double dd = drow[b];
                    if (!((used >> b) & 1) && (best < 0 || dd < bdist)) { best = b; bdist = dd; }
                }
                used |= 1u << best;
                put(best);
            }
        }
    };

    if (SCN == MRB_PCP) {
        const int P = c.num_prey;
        uint32_t sensed = (uint32_t)sci[0], captured = (uint32_t)sci[S];
        const int unseen0 = P - __popc(sensed), left0 = P - __popc(captured);
        double bd = -1.0, bx = -5.0, by = -5.0;
        const bool pred = lane < c.num_predators;
        for (int q = 0; q < P; q++) {
            if ((captured >> q) & 1) continue;
            const double qxp = scf[(2 * q) * S], qyp = scf[(2 * q + 1) * S];
            const double dx = px - qxp, dy = py - qyp, d2 = dx * dx + dy * dy;
            const bool in_range = me && d2 <= (pred ? p.sense_thr2 : 0.0);
            const bool sense = __any_sync(kFull, in_range);
            const bool capture = __any_sync(kFull, me && act == 4 && d2 <= (pred ? 0.0 : p.capture_thr2));
            if (sense) sensed |= 1u << q;
            if (((sensed >> q) & 1) && capture) { captured |= 1u << q; continue; }
            if (in_range) {                                 // rounded norms, strict <: agent.py:32-36, misc.py:14-18
                const double dd = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
                if (bd < 0.0 || dd < bd) { bd = dd; bx = qxp; by = qyp; }
            }
        }
        const int unseen = P - __popc(sensed), left = P - __popc(captured);
        if (lane == 0) { sci[0] = (int32_t)sensed; sci[S] = (int32_t)captured; }
        const int od = c.capability_aware ? 6 : 4;
        int slot = 0;
        if (me) { sbx[lane] = bx; sby[lane] = by; }
        __syncwarp();
        auto put = [&](int b) {
            const ObsRow o(obs, obs64, slot * od);
            o.put(0, spx[b]); o.put(1, spy[b]); o.put(2, sbx[b]); o.put(3, sby[b]);
            if (od == 6) {
                o.put(4, b < c.num_predators ? c.predator_radius : 0.0);
                o.put(5, b < c.num_predators ? 0.0 : c.capture_radius);
            }
            slot++;
        };
        if (me) for_each_block(put);
        if (msg) { rew = c.violation_reward; done = true; }
        else {
            rew = ((unseen0 - unseen) * c.sense_reward + (left0 - left) * c.capture_reward) + c.time_penalty;
            done = steps > c.max_episode_steps || left == 0;
        }
        remaining = left; scen_metric = P - left;
    } else if (SCN == MRB_WAREHOUSE) {
        uint32_t loaded = (uint32_t)sci[0];
        int slot = 0;
        auto put = [&](int b) {
            const ObsRow o(obs, obs64, slot * 3);
            o.put(0, spx[b]); o.put(1, spy[b]); o.put(2, (double)((loaded >> b) & 1));
            slot++;
        };
        if (me) for_each_block(put);
        bool set_bit = false, clr_bit = false;
        if (msg) { rew = c.violation_reward; done = true; }
        else {
            if (me) {
                const bool green = (lane % 2 == 0), ld = (loaded >> lane) & 1;
                if (ld) {
                    if (px < -1.5 + c.goal_width && ((green && py > 0) || (!green && py <= 0))) { rew = c.unload_reward; clr_bit = true; }
                } else {
                    if (px > 1.5 - c.goal_width && ((!green && py > 0) || (green && py <= 0))) { rew = c.load_reward; set_bit = true; }
                }
            }
            done = steps > c.max_episode_steps;
        }
        const uint32_t setm = __ballot_sync(kFull, set_bit), clrm = __ballot_sync(kFull, clr_bit);
        loaded = (loaded | setm) & ~clrm;
        scen_metric = __popc(clrm);
        if (lane == 0) sci[0] = (int32_t)loaded;
    } else if (SCN == MRB_MATERIAL) {
        int load = me ? sci[lane * S] : 0;
        int zone0 = sci[N * S], zone1 = sci[(N + 1) * S];
        int messages = 0;
        for (int i = 0; i < 4; i++) messages |= (__shfl_sync(kFull, act, i) % 4) << (2 * i);
        if (me) {
            const ObsRow o(obs, obs64, 0);
            o.put(0, px); o.put(1, py); o.put(2, (double)load); o.put(3, (double)zone0); o.put(4, (double)zone1);
            for (int i = 0; i < 4; i++) o.put(5 + i, (double)((messages >> (2 * i)) & 3));
            if (c.capability_aware) {
                o.put(9, (double)(lane < c.n_fast ? c.small_torque : c.large_torque));
                o.put(10, lane < c.n_fast ? c.fast_step : c.slow_step);
            }
        }
        double r;
        if (msg) { r = c.violation_reward; done = true; }
        else {
            r = c.time_penalty;
            for (int a = 0; a < N; a++) {               // sequential through the shared zone loads; every lane runs it
                const double xa = __shfl_sync(kFull, px, a), ya = __shfl_sync(kFull, py, a);
                int la = __shfl_sync(kFull, load, a);
                const int torque = a < c.n_fast ? c.small_torque : c.large_torque;
                if (la > 0) {
                    if (xa < -1.5 + c.goal_width) { r += la * c.unload_reward; scen_metric += la; la = 0; }
                } else {
                    int zi = -1;
                    if (xa > 1.5 - c.goal_width) zi = 1;
                    else if (xa * xa + ya * ya <= p.zone1_thr2) zi = 0;
                    if (zi >= 0) {
                        const int zl = zi ? zone1 : zone0, take = zl > torque ? torque : zl;
                        la = take;
                        if (zi) zone1 = zl - take; else zone0 = zl - take;
                        r += take * c.load_reward;
                    }
                }
                if (lane == a) load = la;
            }
            done = steps > c.max_episode_steps;
            if (!done) done = zone0 == 0 && zone1 == 0 && !__any_sync(kFull, me && load != 0);
        }
        rew = r;
        int tot = load;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(kFull, tot, o);
        remaining = zone0 + zone1 + tot;
        if (me) sci[lane * S] = load;
        if (lane == 0) { sci[N * S] = zone0; sci[(N + 1) * S] = zone1; sci[(N + 2) * S] = messages; }
    } else {                                            // Simple
        const double goalx = scf[0], goaly = scf[S];
        if (me) {
            const ObsRow o(obs, obs64, 0);
            int k = 0;
            o.put(k++, px); o.put(k++, py);
            for (int b = 0; b < N; b++) if (b != lane) { o.put(k++, spx[b]); o.put(k++, spy[b]); }
            o.put(k, goalx); o.put(k + 1, goaly);
        }
        const double dx = px - goalx, dy = py - goaly;
        rew = msg ? c.violation_reward : -(dx * dx + dy * dy) * c.reward_scaler;
        done = msg != 0 || steps > c.max_episode_steps;
    }

    // ---------------------------------------------------------------- write back
    if (me) {
        sf[lane * S] = px; sf[(N + lane) * S] = py; sf[(2 * N + lane) * S] = th;
        sf[(3 * N + lane) * S] = qx; sf[(4 * N + lane) * S] = qy;
        p.buf.reward[env * N + lane] = (float)rew;
        if (p.buf.reward_f64) p.buf.reward_f64[env * N + lane] = rew;
        if (p.buf.dist) p.buf.dist[env * N + lane] = (float)dist;
    }
    if (p.hout.obs) {                       // host mirror of this env's observation block (see step_thread.cuh)
        __syncwarp();
        const int64_t base = env * (int64_t)(N * D);
        const int words = N * D;
        if (((base | words) & 3) == 0) {
            const float4 *s4 = reinterpret_cast<const float4 *>(p.buf.obs + base);
            float4 *d4 = reinterpret_cast<float4 *>(p.hout.obs + base);
            for (int k = lane; k < words / 4; k += 32) d4[k] = s4[k];
        } else {
            for (int k = lane; k < words; k += 32) p.hout.obs[base + k] = p.buf.obs[base + k];
        }
    }
    if (me && p.hout.reward) p.hout.reward[env * N + lane] = (float)rew;
    float team = me ? (float)rew : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) team += __shfl_xor_sync(kFull, team, o);
    double ep_return = 0.0;
    if (lane == 0) {
        si[0] = steps; si[S] = 1;
        p.buf.done[env] = done ? 1 : 0;
        p.buf.message[env] = (uint8_t)msg;
        if (p.hout.done) p.hout.done[env] = done ? 1 : 0;
        if (p.hout.message) p.hout.message[env] = (uint8_t)msg;
        p.buf.remaining[env] = remaining;
        ep_return = sf[(5 * N) * S] + (double)team;
        sf[(5 * N) * S] = ep_return;
        if (c.collect_stats && p.buf.stats) {
            double *st = p.buf.stats;
            atomicAdd(st + MRB_STAT_ENV_STEPS, 1.0);
            atomicAdd(st + MRB_STAT_QP_SOLVES, (double)n_qp);
            atomicAdd(st + MRB_STAT_QP_ITERS, (double)n_it);
            atomicAdd(st + MRB_STAT_QP_ITERS_WARP, (double)n_it);       // one env per warp: nothing to wait for
            atomicAdd(st + MRB_STAT_SUBSTEPS, (double)n_sub);
            if (n_stall) atomicAdd(st + MRB_STAT_QP_STALLS, (double)n_stall);
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
    }
    __syncwarp();
    if (done && c.auto_reset && lane == 0) reset_env<SCN>(p, env, si[2 * S]);
}

// MRB_WARP_GENERIC (any value): every team of 7 or more robots runs on the run-time team size kernels, the reference of
// the tensor-core kernels.  Read on every launch: tests switch it within one process.
inline bool warp_generic() { return std::getenv("MRB_WARP_GENERIC") != nullptr; }

// launch(std::integral_constant<int, PPL>()) with the pair slots per lane of N robots rounded up to an instantiated width
template <typename F>
cudaError_t with_runtime_ppl(int N, F &&launch)
{
    const int ppl = team_ppl(N);
    if (ppl <= 1) return launch(std::integral_constant<int, 1>());
    if (ppl <= 2) return launch(std::integral_constant<int, 2>());
    if (ppl <= 4) return launch(std::integral_constant<int, 4>());
    if (ppl <= 6) return launch(std::integral_constant<int, 6>());
    if (ppl <= 8) return launch(std::integral_constant<int, 8>());
    return launch(std::integral_constant<int, 16>());
}

template <int SCN, int PPL, int NC = 0, bool EXACT = true>
inline cudaError_t launch_step_warp_ppl(const Params &p, const int32_t *actions, cudaStream_t s)
{
    constexpr int WPB = NC != 0 ? team_warps(NC) : kWarpsPerBlock;
    const size_t smem = warp_workspace_doubles(NC ? NC : p.cfg.num_robots) * sizeof(double) * WPB;
    const auto kernel = p.envs ? step_warp_kernel<SCN, PPL, NC, WPB, EXACT, true> : step_warp_kernel<SCN, PPL, NC, WPB, EXACT>;
    cudaError_t st = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (st != cudaSuccess) return st;
    const unsigned grid = (unsigned)((p.env_hi - p.env_lo + WPB - 1) / WPB);
    kernel<<<grid, WPB * 32, smem, s>>>(p, actions);
    return cudaSuccess;
}

// Teams of 2..6 robots: one env per thread; 7..32 robots: one env per warp, on the kernel of the scenario's compile-time
// team size (kern_team_*.cu, tensor-core solver; measured against the run-time size in DESIGN.md section 4) where there
// is one, else on the run-time team size kernel.  Explicitly instantiated in kern_step_<scenario>.cu.
template <int SCN>
cudaError_t launch_step(const Params &p, const int32_t *actions, cudaStream_t s)
{
    const int N = p.cfg.num_robots;
    if constexpr (SCN == MRB_ARCTIC) {           // per-terrain step sizes and grid observations, for exactly 4 robots
        return N == 4 ? launch_thread<SCN, 4>(p, actions, s) : cudaErrorNotSupported;
    } else {
        switch (N) {
        case 2: if constexpr (SCN != MRB_MATERIAL) return launch_thread<SCN, 2>(p, actions, s); break;   // MaterialTransport: 4 or more
        case 3: if constexpr (SCN != MRB_MATERIAL) return launch_thread<SCN, 3>(p, actions, s); break;
        case 4: return launch_thread<SCN, 4>(p, actions, s);
        case 5: return launch_thread<SCN, 5>(p, actions, s);
        case 6: return launch_thread<SCN, 6>(p, actions, s);
        default:
            if (team_size(N) <= team_kernel_max(SCN) && !warp_generic())
                return with_team_size<team_kernel_max(SCN)>(N, [&](auto nc) { return launch_step_team<SCN, nc>(p, actions, s, N == nc); });
            return with_runtime_ppl(N, [&](auto ppl) { return launch_step_warp_ppl<SCN, ppl>(p, actions, s); });
        }
        return cudaErrorNotSupported;
    }
}

// ---- barrier QP alone, one problem per warp
template <int PPL, int NC = 0, bool EXACT = true>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, kWarpMinBlocks)
qp_warp_kernel(int N_, int64_t B, int barrier_default, const double *__restrict__ dxi, const double *__restrict__ xi,
               double *__restrict__ u, int32_t *__restrict__ iters)
{
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t e = (int64_t)blockIdx.x * kWarpsPerBlock + wib;
    if (e >= B) return;
    const int N = (NC && EXACT) ? NC : N_;
    QpWarp<PPL, NC, EXACT> qp(N, smem + (size_t)wib * warp_workspace_doubles(NC ? NC : N), lane);
    double xx = 0, xy = 0, ux = 0, uy = 0;
    if (lane < N) { xx = xi[lane * B + e]; xy = xi[(N + lane) * B + e]; ux = dxi[lane * B + e]; uy = dxi[(N + lane) * B + e]; }
    const int it = qp.run(xx, xy, ux, uy, barrier_default != 0);
    if (lane < N) { u[lane * B + e] = ux; u[(N + lane) * B + e] = uy; }
    if (iters && lane == 0) iters[e] = it;
}

template <int PPL, int NC = 0, bool EXACT = true>
inline cudaError_t launch_qp_warp_ppl(int N, int bd, int64_t B, const double *dxi, const double *xi, double *u, int32_t *iters, cudaStream_t s)
{
    const size_t smem = warp_workspace_doubles(NC ? NC : N) * sizeof(double) * kWarpsPerBlock;
    cudaError_t st = cudaFuncSetAttribute(qp_warp_kernel<PPL, NC, EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (st != cudaSuccess) return st;
    qp_warp_kernel<PPL, NC, EXACT><<<(unsigned)((B + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, smem, s>>>(N, B, bd, dxi, xi, u, iters);
    return cudaSuccess;
}

}  // namespace mrb
