// Barrier-certificate QP, one env per thread, primal normal equations (teams of 5 and 6 robots).
//
// Replaces rps create_single_integrator_barrier_certificate{,2} -> cvxopt.solvers.qp (called at
// /root/reference/robotarium_gym/utilities/controller.py:23; SURVEY.md App. A.8 / A.9).
// The iteration is cvxopt's coneqp for a pure 'l' cone (Mehrotra predictor-corrector, STEP 0.99,
// EXPON 3, default start, rps' options reltol = feastol = 1e-2, abstol 1e-7, maxiters 50) with
// cvxopt's data-dependent stopping rule, written in UNscaled variables: for the 'l' cone the
// Nesterov-Todd scaling W = diag(sqrt(s/z)) cancels algebraically, so (dx, ds, dz), the step
// lengths and sigma are the same numbers up to rounding.
//
// Structure that is exploited instead of a dense G (m x 2N):
//   row c = pair (i<j):  g_c = [ -a_c at block i, +a_c at block j ],  a_c = 2 (xi_i - xi_j) in R^2
//   (G v)_c = a_c . (v_j - v_i);  G'y scatters -+ a_c y_c;  K = 2I + G' diag(w) G is a weighted
//   graph Laplacian of 2x2 blocks  w_c a_c a_c'  -> packed lower-triangular Cholesky, no pivoting.
#pragma once
#include "common.cuh"

namespace mrb {

// Storage.  Registers cap the number of resident warps, and these kernels are bound by dependent-issue latency, i.e.
// by how many warps an SM sub-partition can switch between (DESIGN.md section 4).  The 2N x 2N Cholesky factor is kept
// as N x N blocks of 2 x 2 (one block per robot pair, [e0 e1; e2 e3] = rows 2a, 2a+1 x columns 2b, 2b+1).  The
// diagonal blocks live in registers as (1/l11, 1/l22, l21).  The strictly-lower blocks live in SHARED memory, two
// 128-bit words per block, interleaved over the threads of the CTA (word w of thread t at Ls[w * TPB + t]:
// conflict-free).  With everything in registers a 6-robot team needs ~350 live doubles per env and the kernel spills
// ~1.9 KB per thread to local memory; the factor is the one large array whose accesses are few enough per flop (each
// block is read once per triangular solve, and the block-row factorisation below reads 20 blocks and writes 15) to
// sit behind the 128 B/clk shared-memory pipe.  Two per-constraint vectors (m = N(N-1)/2 numbers each), h and rz,
// live in the same store, one double per constraint interleaved over the threads like the factor; the other vectors
// are register arrays.

// One per-env vector in the shared store: element c of this thread's vector at base[c * TPB].
template <int TPB>
struct SharedCol {
    double *base;
    // volatile: without it the compiler merges the repeated loads of one iteration into a single early load and
    // keeps the value live (then spills it to local memory) -- the opposite of what this store is for
    __device__ __forceinline__ double get(int c) const { return reinterpret_cast<const volatile double *>(base)[c * TPB]; }
    __device__ __forceinline__ void set(int c, double v) { reinterpret_cast<volatile double *>(base)[c * TPB] = v; }
};
__device__ __forceinline__ void lds_block(uint32_t addr, uint32_t stride, double (&o)[4])
{
    asm volatile("ld.volatile.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o[0]), "=d"(o[1]) : "r"(addr));
    asm volatile("ld.volatile.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o[2]), "=d"(o[3]) : "r"(addr + stride));
}
__device__ __forceinline__ void sts_block(uint32_t addr, uint32_t stride, const double (&o)[4])
{
    asm volatile("st.volatile.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(o[0]), "d"(o[1]));
    asm volatile("st.volatile.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr + stride), "d"(o[2]), "d"(o[3]));
}

// TPB: threads per CTA (the interleave stride of the shared store)
template <int N, int TPB>
struct QpThread {
    static constexpr int n = 2 * N;
    static constexpr int m = N * (N - 1) / 2;
    __device__ static constexpr int lowidx(int a, int b) { return a * (a - 1) / 2 + b; }        // a > b
    static constexpr int kSmemWords = 2 * m;                      // factor: double2 words per thread (m blocks)
    static constexpr int kVecDoubles = 2 * m;                     // h, rz: doubles per thread
    __device__ static constexpr int pair(int i, int j) { return i * (2 * N - i - 1) / 2 + (j - i - 1); }   // i < j

    double ax[m], ay[m];
    double invd[n], l21[N];
    uint32_t Ls;                 // shared-window address of this thread's first factor word
    double *Vs;                  // this thread's first vector double

    template <int A, int B>
    __device__ __forceinline__ void load_blk(double (&o)[4]) const
    {
        lds_block(Ls + (2 * lowidx(A, B)) * TPB * 16, TPB * 16, o);
    }
    template <int A, int B>
    __device__ __forceinline__ void store_blk(const double (&o)[4])
    {
        sts_block(Ls + (2 * lowidx(A, B)) * TPB * 16, TPB * 16, o);
    }

    __device__ __forceinline__ QpThread(double2 *Ls_, double *Vs_) : Ls((uint32_t)__cvta_generic_to_shared(Ls_)), Vs(Vs_) {}

    // sink(c, (G v)_c) for every constraint c
    template <typename F>
    __device__ __forceinline__ void G_mul(const double (&v)[n], F &&sink) const
    {
        int c = 0;
#pragma unroll
        for (int i = 0; i < N - 1; i++)
#pragma unroll
            for (int j = i + 1; j < N; j++, c++)
                sink(c, ax[c] * (v[2 * j] - v[2 * i]) + ay[c] * (v[2 * j + 1] - v[2 * i + 1]));
    }
    // out += G' y,  y given as a function of the constraint index
    template <typename F>
    __device__ __forceinline__ void GT_acc(F &&y, double (&out)[n]) const
    {
        int c = 0;
#pragma unroll
        for (int i = 0; i < N - 1; i++)
#pragma unroll
            for (int j = i + 1; j < N; j++, c++) {
                const double yc = y(c);
                const double tx = ax[c] * yc, ty = ay[c] * yc;
                out[2 * i] -= tx; out[2 * i + 1] -= ty;
                out[2 * j] += tx; out[2 * j + 1] += ty;
            }
    }
    // L := chol(2I + G' diag(w) G), one block row at a time (bordering): block row a is built in registers
    // from the rows above it, L_ab = (K_ab - sum_{c<b} L_ac L_bc') L_bb^-T, then the diagonal block from
    // K_aa - sum_c L_ac L_ac'.  K is never stored: K_ab = -w_c a_c a_c' for the pair c = (b, a).
    template <typename W>
    __device__ __forceinline__ void factor(W &&w)
    {
        double dxx[N], dxy[N], dyy[N];
#pragma unroll
        for (int a = 0; a < N; a++) { dxx[a] = 2.0; dxy[a] = 0.0; dyy[a] = 2.0; }
        {
            int c = 0;
#pragma unroll
            for (int i = 0; i < N - 1; i++)
#pragma unroll
                for (int j = i + 1; j < N; j++, c++) {
                    const double wc = w(c), ac = ax[c], bc = ay[c];
                    const double wx = wc * ac, wy = wc * bc;
                    const double pxx = wx * ac, pxy = wx * bc, pyy = wy * bc;
                    dxx[i] += pxx; dxy[i] += pxy; dyy[i] += pyy;
                    dxx[j] += pxx; dxy[j] += pxy; dyy[j] += pyy;
                }
        }
        static_for<0, N>([&](auto A_) {
            constexpr int a = decltype(A_)::value;
            double R[a > 0 ? a : 1][4] = {};
            static_for<0, a>([&](auto B_) {
                constexpr int b = decltype(B_)::value;
                constexpr int c = pair(b, a);
                const double wc = w(c), ac = ax[c], bc = ay[c];
                const double wx = wc * ac, wy = wc * bc;
                double s0 = -wx * ac, s1 = -wx * bc, s2 = s1, s3 = -wy * bc;
                static_for<0, b>([&](auto C_) {
                    constexpr int cc = decltype(C_)::value;
                    double T[4];
                    load_blk<b, cc>(T);
                    s0 = fma(-R[cc][0], T[0], s0); s0 = fma(-R[cc][1], T[1], s0);
                    s1 = fma(-R[cc][0], T[2], s1); s1 = fma(-R[cc][1], T[3], s1);
                    s2 = fma(-R[cc][2], T[0], s2); s2 = fma(-R[cc][3], T[1], s2);
                    s3 = fma(-R[cc][2], T[2], s3); s3 = fma(-R[cc][3], T[3], s3);
                });
                const double r1 = invd[2 * b], r2 = invd[2 * b + 1], lo = l21[b];
                R[b][0] = s0 * r1; R[b][2] = s2 * r1;
                R[b][1] = fma(-R[b][0], lo, s1) * r2;
                R[b][3] = fma(-R[b][2], lo, s3) * r2;
            });
            double d0 = dxx[a], d1 = dxy[a], d2 = dyy[a];
#pragma unroll
            for (int b = 0; b < a; b++) {
                d0 = fma(-R[b][0], R[b][0], d0); d0 = fma(-R[b][1], R[b][1], d0);
                d1 = fma(-R[b][2], R[b][0], d1); d1 = fma(-R[b][3], R[b][1], d1);
                d2 = fma(-R[b][2], R[b][2], d2); d2 = fma(-R[b][3], R[b][3], d2);
            }
            const double r1 = fast_rsqrt(d0);
            const double lo = d1 * r1;
            const double r2 = fast_rsqrt(fma(-lo, lo, d2));
            invd[2 * a] = r1; invd[2 * a + 1] = r2; l21[a] = lo;
            static_for<0, a>([&](auto B_) {
                constexpr int b = decltype(B_)::value;
                store_blk<a, b>(R[b]);
            });
        });
    }
    // v := K^-1 v: block forward substitution, then block backward substitution in row order (after x_a is
    // known, every earlier block row receives -L_ab' x_a), so each stored block is read once per sweep
    __device__ __forceinline__ void solve(double (&v)[n]) const
    {
        static_for<0, N>([&](auto A_) {
            constexpr int a = decltype(A_)::value;
            double bx = v[2 * a], by = v[2 * a + 1];
            static_for<0, a>([&](auto B_) {
                constexpr int b = decltype(B_)::value;
                double T[4];
                load_blk<a, b>(T);
                bx = fma(-T[0], v[2 * b], bx); bx = fma(-T[1], v[2 * b + 1], bx);
                by = fma(-T[2], v[2 * b], by); by = fma(-T[3], v[2 * b + 1], by);
            });
            const double y0 = bx * invd[2 * a];
            v[2 * a] = y0;
            v[2 * a + 1] = fma(-l21[a], y0, by) * invd[2 * a + 1];
        });
        static_for<0, N>([&](auto A_) {
            constexpr int a = N - 1 - decltype(A_)::value;
            const double x1 = v[2 * a + 1] * invd[2 * a + 1];
            const double x0 = fma(-l21[a], x1, v[2 * a]) * invd[2 * a];
            v[2 * a] = x0; v[2 * a + 1] = x1;
            static_for<0, a>([&](auto B_) {
                constexpr int b = decltype(B_)::value;
                double T[4];
                load_blk<a, b>(T);
                v[2 * b] = fma(-T[0], x0, v[2 * b]); v[2 * b] = fma(-T[2], x1, v[2 * b]);
                v[2 * b + 1] = fma(-T[1], x0, v[2 * b + 1]); v[2 * b + 1] = fma(-T[3], x1, v[2 * b + 1]);
            });
        });
    }

    // xi: SI points; u: in = nominal dxi (already norm-limited to 0.15 by the position controller),
    // out = certified velocities.  Returns the number of interior-point iterations.
    __device__ __forceinline__ int run(const double (&xix)[N], const double (&xiy)[N], double (&ux)[N], double (&uy)[N],
                                       bool barrier_default)
    {
        double q[n], x[n];
#pragma unroll
        for (int i = 0; i < N; i++) {          // A.8: pre-clip columns of dxi to norm 0.2, f = -2 dxi
            double nrm = sqrt(ux[i] * ux[i] + uy[i] * uy[i]);
            if (nrm > kQpMagnitudeLimit) {
                double sc = kQpMagnitudeLimit / nrm;
                ux[i] *= sc; uy[i] *= sc;
            }
            q[2 * i] = -2.0 * ux[i];
            q[2 * i + 1] = -2.0 * uy[i];
        }
        SharedCol<TPB> h{Vs}, rz{Vs + (size_t)m * TPB};
        double s[m], z[m], t2[m], w[m];

        const double r2 = barrier_default ? 0.17 * 0.17 : 0.2 * 0.2;
        double hh = 0.0, qq = 0.0;
        {
            int c = 0;
#pragma unroll
            for (int i = 0; i < N - 1; i++)
#pragma unroll
                for (int j = i + 1; j < N; j++, c++) {
                    double ex = xix[i] - xix[j], ey = xiy[i] - xiy[j];
                    double hv = (ex * ex + ey * ey) - r2;
                    double gain = barrier_default ? 100.0 : (hv >= 0.0 ? 100.0 : 1e6);
                    const double hc = gain * (hv * hv * hv);
                    h.set(c, hc);
                    ax[c] = 2.0 * ex; ay[c] = 2.0 * ey;
                    hh += hc * hc;
                }
#pragma unroll
            for (int a = 0; a < n; a++) qq += q[a] * q[a];
        }
        const double feas_x2 = 1e-4 * dmax(qq, 1.0), feas_z2 = 1e-4 * dmax(hh, 1.0);

        // ---- default starting point: (2I + G'G) x = -q + G'h ; z = Gx - h ; s = -z ; shift
        factor([](int) { return 1.0; });
#pragma unroll
        for (int a = 0; a < n; a++) x[a] = -q[a];
        GT_acc([&](int c) { return h.get(c); }, x);
        solve(x);
        double ss = 0.0, ts = -INFINITY, tz = -INFINITY;
        G_mul(x, [&](int c, double gx) {
            const double zc = gx - h.get(c);
            z[c] = zc;
            ss += zc * zc;
            ts = dmax(zc, ts);                // max(-s) = max(z)
            tz = dmax(-zc, tz);
        });
        const double nrm = ss > 1.0 ? ss * fast_rsqrt(ss) : 1.0;          // max(|z|, 1)
        const double s_shift = ts >= -1e-8 * nrm ? 1.0 + ts : 0.0, z_shift = tz >= -1e-8 * nrm ? 1.0 + tz : 0.0;
        const bool do_s = ts >= -1e-8 * nrm, do_z = tz >= -1e-8 * nrm;
        double gap = 0.0;
#pragma unroll
        for (int c = 0; c < m; c++) {
            const double z0 = z[c];
            double sc = -z0, zc = z0;
            if (do_s) sc += s_shift;
            if (do_z) zc += z_shift;
            s[c] = sc; z[c] = zc;
            gap += sc * zc;
        }

        int iters = 0;
        for (; iters <= 50; iters++) {
            double rx[n];
            // rx = 2x + q + G'z ; f0 = 1/2 x'Px + q'x ; rz = s + Gx - h
            double xq = 0.0, xrx = 0.0;
#pragma unroll
            for (int a = 0; a < n; a++) {
                rx[a] = 2.0 * x[a] + q[a];
                xrx += x[a] * rx[a];
                xq += x[a] * q[a];
            }
            const double f0 = 0.5 * (xrx + xq);
            GT_acc([&](int c) { return z[c]; }, rx);
            double resx = 0.0, resx1 = 0.0, resz = 0.0, resz1 = 0.0, zrz = 0.0, zrz1 = 0.0;      // sums in two halves
#pragma unroll
            for (int a = 0; a < n; a += 2) { resx = fma(rx[a], rx[a], resx); resx1 = fma(rx[a + 1], rx[a + 1], resx1); }
            resx += resx1;
            G_mul(x, [&](int c, double gx) {
                const double r = gx + (s[c] - h.get(c));
                rz.set(c, r);
                if (c & 1) { resz1 = fma(r, r, resz1); zrz1 = fma(z[c], r, zrz1); }
                else { resz = fma(r, r, resz); zrz = fma(z[c], r, zrz); }
            });
            resz += resz1; zrz += zrz1;
            const double pcost = f0, dcost = f0 + zrz - gap;
            bool gap_ok = gap <= 1e-7;
            if (pcost < 0.0) gap_ok = gap_ok || (gap <= -1e-2 * pcost);
            else if (dcost > 0.0) gap_ok = gap_ok || (gap <= 1e-2 * dcost);
            if ((resz <= feas_z2 && resx <= feas_x2 && gap_ok) || iters == 50) break;

            // w = z/s ; K = 2I + G' diag(w) G
#pragma unroll
            for (int c = 0; c < m; c++) w[c] = z[c] * fast_rcp1(s[c]);
            // 1/s and 1/z are recomputed where they are used (same function of the same input: identical bits), and the
            // corrector's (ds, dz) are recomputed in the update pass instead of being stored: two SFU seeds and ~10 flops
            // per constraint buy four fewer per-constraint vectors to keep on chip
            auto inv_s = [&](int c) { return fast_rcp1(s[c]); };
            auto inv_z = [&](int c) { return fast_rcp1(z[c]); };
            factor([&](int c) { return w[c]; });

            // predictor (rc = -s.z):                 K dx = -rx - G'(w.rz - z)
            // corrector (rc = -s.z - ds_aff.dz_aff + sigma mu):  K dx = -rx - G'(w.rz - z + t2),  t2 = (rc + s.z)/s
            // (running one body twice under a runtime `pass` flag to halve the code was measured 2.5x slower)
            double dx[n];
            double tmax;
            // step-length maximum over the 2m candidates in four interleaved running maxima (depth m/4 + 2 instead of a
            // serial chain of 2m; a full pairwise tree would keep m candidates live, which this kernel has no registers for)
            double tm[4];
#pragma unroll
            for (int a = 0; a < n; a++) dx[a] = -rx[a];
            GT_acc([&](int c) { return z[c] - w[c] * rz.get(c); }, dx);
            solve(dx);
            double dsdz = 0.0, dsdz1 = 0.0;
            tm[0] = tm[1] = tm[2] = tm[3] = 0.0;
            G_mul(dx, [&](int c, double gd) {
                const double dsc = -rz.get(c) - gd;
                const double dzc = -z[c] - w[c] * dsc;
                const double pr = dsc * dzc;                 // Mehrotra correction term
                t2[c] = pr;
                if (c & 1) dsdz1 += pr; else dsdz += pr;
                tm[c & 3] = dmax(dmax(-dsc * inv_s(c), -dzc * inv_z(c)), tm[c & 3]);
            });
            dsdz += dsdz1;
            tmax = dmax(dmax(tm[0], tm[1]), dmax(tm[2], tm[3]));
            double step = tmax <= 1.0 ? 1.0 : fast_rcp(tmax);
            double sg = dmin(dmax(1.0 - step + dsdz * fast_rcp(gap) * (step * step), 0.0), 1.0);
            const double sigmamu = sg * sg * sg * (gap / m);
#pragma unroll
            for (int c = 0; c < m; c++) t2[c] = (sigmamu - t2[c]) * inv_s(c);         // (rc + s.z)/s
#pragma unroll
            for (int a = 0; a < n; a++) dx[a] = -rx[a];
            GT_acc([&](int c) { return z[c] - w[c] * rz.get(c) - t2[c]; }, dx);   // -(rc + z.rz)/s
            solve(dx);
            tm[0] = tm[1] = tm[2] = tm[3] = 0.0;
            G_mul(dx, [&](int c, double gd) {
                const double dsc = -rz.get(c) - gd;
                const double dzc = fma(-w[c], dsc, t2[c] - z[c]);                 // (rc - z.ds)/s
                tm[c & 3] = dmax(dmax(-dsc * inv_s(c), -dzc * inv_z(c)), tm[c & 3]);
            });
            tmax = dmax(dmax(tm[0], tm[1]), dmax(tm[2], tm[3]));
            step = tmax <= 0.99 ? 1.0 : 0.99 * fast_rcp(tmax);
            gap = 0.0;
            double gap1 = 0.0;
            // the same expressions again; dx is laundered so that the compiler does not keep the first pass's
            // 2m results live across the step-length reduction
#pragma unroll
            for (int a = 0; a < n; a++) asm volatile("" : "+d"(dx[a]));
            G_mul(dx, [&](int c, double gd) {
                const double dsc = -rz.get(c) - gd;
                const double zc0 = z[c];
                const double dzc = fma(-w[c], dsc, t2[c] - zc0);
                const double sc = fma(step, dsc, s[c]), zc = fma(step, dzc, zc0);
                s[c] = sc; z[c] = zc;
                if (c & 1) gap1 = fma(sc, zc, gap1); else gap = fma(sc, zc, gap);
            });
            gap += gap1;
#pragma unroll
            for (int a = 0; a < n; a++) x[a] += step * dx[a];
        }
#pragma unroll
        for (int i = 0; i < N; i++) {
            ux[i] = x[2 * i];
            uy[i] = x[2 * i + 1];
        }
        return iters;
    }
};

}  // namespace mrb
