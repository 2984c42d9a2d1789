// The N <= 4 barrier-QP iteration as it was before the LDL' rewrite of qp_dual.cuh (Cholesky factor with an rsqrt per
// pivot, branchy stopping rule, gap / m by division), kept verbatim as the reference that
// tests/test_qp_dual_iteration.py compares the library's QpDual<N> with.  Compiled by that test only.
#include <cstdint>
#include "common.cuh"
#include "qp_dual.cuh"

namespace mrb_ref {
using namespace mrb;

template <int N>
struct QpDualCholesky {
    static constexpr int n = 2 * N;
    static constexpr int m = N * (N - 1) / 2;
    static constexpr int MT = m * (m - 1) / 2;                 // strictly-lower entries
    __device__ static constexpr int low(int r, int c) { return r * (r - 1) / 2 + c; }   // r > c

    double ax[m], ay[m];
    double L[MT];
    double invd[m];

    // sink(c, (G v)_c)
    template <typename V, typename F>
    __device__ __forceinline__ void G_mul(V &&v, F &&sink) const
    {
        int c = 0;
#pragma unroll
        for (int i = 0; i < N - 1; i++)
#pragma unroll
            for (int j = i + 1; j < N; j++, c++)
                sink(c, ax[c] * (v(2 * j) - v(2 * i)) + ay[c] * (v(2 * j + 1) - v(2 * i + 1)));
    }
    // out += G' y
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
    // entry (c, e), e < c, of 1/2 G G': +-(a_c . a_e)/2 when the two pairs share a robot, else 0
    template <int C, int E>
    __device__ __forceinline__ double gram() const
    {
        constexpr int ci = pair_i(C), cj = pair_j(C), ei = pair_i(E), ej = pair_j(E);
        constexpr int sgn = (ci == ei) + (cj == ej) - (ci == ej) - (cj == ei);
        if constexpr (sgn == 0) return 0.0;
        else {
            const double dot = fma(ax[C], ax[E], ay[C] * ay[E]);
            return sgn > 0 ? 0.5 * dot : -0.5 * dot;
        }
    }
    __device__ static constexpr int pair_i(int c) { int i = 0; while (c >= N - 1 - i) { c -= N - 1 - i; i++; } return i; }
    __device__ static constexpr int pair_j(int c) { int i = 0; while (c >= N - 1 - i) { c -= N - 1 - i; i++; } return i + 1 + c; }

    // L := chol(1/2 G G' + diag(d)), column by column (left-looking): pivot k from its own row, then the entries below
    // it, which are independent of each other.  The Gram entries are formed where they are consumed (never stored).
    // Per column the dependent chain is (last product of the sums) -> rsqrt -> scale, 72 cycles, against a chain that
    // grows with the row index in a row-by-row order (measured latencies: profiles/r02_fp64_latency_microbench.txt).
    template <typename D>
    __device__ __forceinline__ void factor(D &&d)
    {
        static_for<0, m>([&](auto K_) {
            constexpr int k = decltype(K_)::value;
            const double a = ax[k], b = ay[k];
            double dk = fma(a, a, b * b) + d(k);                                    // 1/2 |g_k|^2 = |a_k|^2
#pragma unroll
            for (int j = 0; j < k; j++) { const double l = L[low(k, j)]; dk = fma(-l, l, dk); }
            const double r = fast_rsqrt(dk);
            invd[k] = r;
            static_for<k + 1, m>([&](auto I_) {
                constexpr int i = decltype(I_)::value;
                double v = gram<i, k>();
#pragma unroll
                for (int j = 0; j < k; j++) v = fma(-L[low(i, j)], L[low(k, j)], v);
                L[low(i, k)] = v * r;
            });
        });
    }
    // b := (L L')^-1 b
    __device__ __forceinline__ void solve(double (&b)[m]) const
    {
        static_for<0, m>([&](auto I) {
            constexpr int i = decltype(I)::value;
            double v = b[i];
#pragma unroll
            for (int k = 0; k < i; k++) v = fma(-L[low(i, k)], b[k], v);
            b[i] = v * invd[i];
        });
        // backward sweep in row order: once x_i is known every earlier row receives -L_ik x_i
        static_for<0, m>([&](auto I) {
            constexpr int i = m - 1 - decltype(I)::value;
            const double xi = b[i] * invd[i];
            b[i] = xi;
#pragma unroll
            for (int k = 0; k < i; k++) b[k] = fma(-L[low(i, k)], xi, b[k]);
        });
    }

    __device__ __forceinline__ int run(const double (&xix)[N], const double (&xiy)[N], double (&ux)[N],
                                       double (&uy)[N], bool barrier_default)
    {
        double q[n], x[n];
#pragma unroll
        for (int i = 0; i < N; i++) {          // A.8: pre-clip columns of dxi to norm 0.2, f = -2 dxi
            const double n2 = ux[i] * ux[i] + uy[i] * uy[i];
            if (n2 > kQpMagnitudeLimit * kQpMagnitudeLimit) {
                const double sc = kQpMagnitudeLimit / sqrt(n2);
                ux[i] *= sc; uy[i] *= sc;
            }
            q[2 * i] = -2.0 * ux[i];
            q[2 * i + 1] = -2.0 * uy[i];
        }
        double h[m], s[m], z[m], rz[m], rxs[n], t2[m], dd[m], corr[m], pp[m];

        const double r2 = barrier_default ? 0.17 * 0.17 : 0.2 * 0.2;
        double hh = 0.0, qq = 0.0;
        {
            int c = 0;
#pragma unroll
            for (int i = 0; i < N - 1; i++)
#pragma unroll
                for (int j = i + 1; j < N; j++, c++) {
                    const double ex = xix[i] - xix[j], ey = xiy[i] - xiy[j];
                    const double hv = (ex * ex + ey * ey) - r2;
                    const double gain = barrier_default ? 100.0 : (hv >= 0.0 ? 100.0 : 1e6);
                    const double hc = gain * (hv * hv * hv);
                    h[c] = hc;
                    ax[c] = 2.0 * ex; ay[c] = 2.0 * ey;
                    hh = fma(hc, hc, hh);
                }
        }
        {
            double q0 = 0.0, q1 = 0.0;
#pragma unroll
            for (int a = 0; a < n; a += 2) {
                const double qa = q[a], qb = q[a + 1];
                q0 = fma(qa, qa, q0); q1 = fma(qb, qb, q1);
            }
            qq = q0 + q1;
        }
        // (feastol * max(1, |q|))^2 and (feastol * max(1, |h|))^2
        const double feas_x2 = 1e-4 * dmax(qq, 1.0), feas_z2 = 1e-4 * dmax(hh, 1.0);

        // ---- default starting point [P G'; G -I][x; z] = [-q; h]:  (1/2 GG' + I) z = -h - 1/2 G q,  x = -1/2 (q + G'z)
        factor([](int) { return 1.0; });
        double tv[m];
        G_mul([&](int a) { return q[a]; }, [&](int c, double g) { tv[c] = -h[c] - 0.5 * g; });
        solve(tv);
        {
            double xa[n];
#pragma unroll
            for (int a = 0; a < n; a++) xa[a] = q[a];
            GT_acc([&](int c) { return tv[c]; }, xa);
#pragma unroll
            for (int a = 0; a < n; a++) x[a] = xa[a] * -0.5;
        }
        double ss = 0.0, ts = -INFINITY, tz = -INFINITY;
        G_mul([&](int a) { return x[a]; }, [&](int c, double g) {       // z = Gx - h as cvxopt forms it
            const double zc = g - h[c];
            z[c] = zc;
            ss = fma(zc, zc, ss);
            ts = dmax(zc, ts);
            tz = dmax(-zc, tz);
        });
        const double nrm = ss > 1.0 ? ss * fast_rsqrt(ss) : 1.0;          // max(|z|, 1)
        const bool do_s = ts >= -1e-8 * nrm, do_z = tz >= -1e-8 * nrm;
        double gap = 0.0;
#pragma unroll
        for (int c = 0; c < m; c++) {
            const double z0 = z[c];
            double sc = -z0, zc = z0;
            if (do_s) sc += 1.0 + ts;
            if (do_z) zc += 1.0 + tz;
            s[c] = sc; z[c] = zc;
            gap = fma(sc, zc, gap);
        }

        int iters = 0;
        for (; iters <= 50; iters++) {
            double rx[n];
            // the sums of this block are accumulated in two halves each (even / odd terms): half the dependent depth
            double xq = 0.0, xrx = 0.0, xq1 = 0.0, xrx1 = 0.0;
#pragma unroll
            for (int a = 0; a < n; a += 2) {
                const double xa = x[a], qa = q[a], xb = x[a + 1], qb = q[a + 1];
                rx[a] = fma(2.0, xa, qa);
                rx[a + 1] = fma(2.0, xb, qb);
                xrx = fma(xa, rx[a], xrx); xrx1 = fma(xb, rx[a + 1], xrx1);
                xq = fma(xa, qa, xq); xq1 = fma(xb, qb, xq1);
            }
            const double f0 = 0.5 * ((xrx + xrx1) + (xq + xq1));
            GT_acc([&](int c) { return z[c]; }, rx);
            double resx = 0.0, resx1 = 0.0, resz = 0.0, resz1 = 0.0, zrz = 0.0, zrz1 = 0.0;
#pragma unroll
            for (int a = 0; a < n; a += 2) { resx = fma(rx[a], rx[a], resx); resx1 = fma(rx[a + 1], rx[a + 1], resx1); }
            resx += resx1;
            G_mul([&](int a) { return x[a]; }, [&](int c, double g) {
                const double r = g + (s[c] - h[c]);
                rz[c] = r;
                if (c & 1) { resz1 = fma(r, r, resz1); zrz1 = fma(z[c], r, zrz1); }
                else { resz = fma(r, r, resz); zrz = fma(z[c], r, zrz); }
            });
            resz += resz1; zrz += zrz1;
            const double pcost = f0, dcost = f0 + zrz - gap;
            // cvxopt's stopping rule without sqrt / division: relgap <= reltol  <=>  gap <= 1e-2 * denominator,
            // pres = sqrt(resz)/resz0 <= feastol  <=>  resz <= (1e-2 * resz0)^2   (equal up to 1 ulp at the threshold)
            bool gap_ok = gap <= 1e-7;
            if (pcost < 0.0) gap_ok = gap_ok || (gap <= -1e-2 * pcost);
            else if (dcost > 0.0) gap_ok = gap_ok || (gap <= 1e-2 * dcost);
            if ((resz <= feas_z2 && resx <= feas_x2 && gap_ok) || iters == 50) break;

            // 1/s and 1/z are recomputed where they are used (same function of the same input: identical bits)
            auto inv_s = [&](int c) { return fast_rcp1(s[c]); };
            auto inv_z = [&](int c) { return fast_rcp1(z[c]); };
#pragma unroll
            for (int c = 0; c < m; c++) dd[c] = s[c] * inv_z(c);           // D = s/z
            factor([&](int c) { return dd[c]; });
            // base right-hand side shared by predictor and corrector: rz - 1/2 G rx - s
            G_mul([&](int a) { return rx[a]; }, [&](int c, double g) { t2[c] = rz[c] - 0.5 * g - s[c]; });
#pragma unroll
            for (int a = 0; a < n; a++) rxs[a] = rx[a];                          // rx is needed again after the solves
            // predictor (rc = -s.z)
            double dz[m];
#pragma unroll
            for (int c = 0; c < m; c++) dz[c] = t2[c];
            solve(dz);
            double dsdz = 0.0, dsdz1 = 0.0, tmax;
            double cand[m];
#pragma unroll
            for (int c = 0; c < m; c++) {
                const double sc = s[c];
                const double dsc = -sc - dd[c] * dz[c];
                const double p = dsc * dz[c];
                if (c & 1) dsdz1 += p; else dsdz += p;
                cand[c] = dmax(-dsc * inv_s(c), -dz[c] * inv_z(c));
                pp[c] = p;                                  // keep only the Mehrotra correction term
            }
            dsdz += dsdz1;
            tmax = dmax(tree_max(cand), 0.0);
            double step = tmax <= 1.0 ? 1.0 : fast_rcp(tmax);          // t == 0 ? 1 : min(1, 1/t)
            const double sg = dmin(dmax(1.0 - step + dsdz * fast_rcp(gap) * (step * step), 0.0), 1.0);
            const double sigmamu = sg * sg * sg * (gap / m);
            // corrector (rc = -s.z - ds_aff.dz_aff + sigma mu)
#pragma unroll
            for (int c = 0; c < m; c++) {
                const double cr = (sigmamu - pp[c]) * inv_z(c);        // (rc + s.z)/z
                corr[c] = cr;
                dz[c] = t2[c] + cr;
            }
            solve(dz);
#pragma unroll
            for (int c = 0; c < m; c++) {
                const double dsc = corr[c] - s[c] - dd[c] * dz[c];
                cand[c] = dmax(-dsc * inv_s(c), -dz[c] * inv_z(c));
            }
            tmax = dmax(tree_max(cand), 0.0);
            step = tmax <= 0.99 ? 1.0 : 0.99 * fast_rcp(tmax);          // t == 0 ? 1 : min(1, 0.99/t)
            // dx = -1/2 (rx + G'dz)
            double rx2[n];
#pragma unroll
            for (int a = 0; a < n; a++) rx2[a] = rxs[a];
            GT_acc([&](int c) { return dz[c]; }, rx2);
            const double hstep = -0.5 * step;
#pragma unroll
            for (int a = 0; a < n; a++) x[a] = fma(hstep, rx2[a], x[a]);
            gap = 0.0;
            double gap1 = 0.0;
#pragma unroll
            for (int c = 0; c < m; c++) {
                const double s0 = s[c];
                const double dsc = corr[c] - s0 - dd[c] * dz[c];
                const double sc = fma(step, dsc, s0), zc = fma(step, dz[c], z[c]);
                s[c] = sc; z[c] = zc;
                if (c & 1) gap1 = fma(sc, zc, gap1); else gap = fma(sc, zc, gap);
            }
            gap += gap1;
        }
#pragma unroll
        for (int i = 0; i < N; i++) {
            ux[i] = x[2 * i];
            uy[i] = x[2 * i + 1];
        }
        return iters;
    }
};


// one problem per thread, both iterations on the same input; layout as mrb_barrier_qp: xi, dxi, u are [2N, B]
template <int N>
__global__ void both_kernel(int64_t B, int barrier_default, const double *__restrict__ dxi, const double *__restrict__ xi,
                            double *__restrict__ u_ref, int32_t *__restrict__ it_ref, double *__restrict__ u_new,
                            int32_t *__restrict__ it_new)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    double xix[N], xiy[N], ux[N], uy[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
        xix[i] = xi[i * B + e]; xiy[i] = xi[(N + i) * B + e];
        ux[i] = dxi[i * B + e]; uy[i] = dxi[(N + i) * B + e];
    }
    {
        double vx[N], vy[N];
        for (int i = 0; i < N; i++) { vx[i] = ux[i]; vy[i] = uy[i]; }
        QpDualCholesky<N> qp;
        it_ref[e] = qp.run(xix, xiy, vx, vy, barrier_default != 0);
        for (int i = 0; i < N; i++) { u_ref[i * B + e] = vx[i]; u_ref[(N + i) * B + e] = vy[i]; }
    }
    {
        QpDual<N> qp;
        it_new[e] = qp.run(xix, xiy, ux, uy, barrier_default != 0);
        for (int i = 0; i < N; i++) { u_new[i * B + e] = ux[i]; u_new[(N + i) * B + e] = uy[i]; }
    }
}

}  // namespace mrb_ref

extern "C" int qp_both(int N, int barrier_default, int64_t B, const double *dxi, const double *xi, double *u_ref,
                       int32_t *it_ref, double *u_new, int32_t *it_new)
{
    const int tpb = 64;
    const unsigned grid = (unsigned)((B + tpb - 1) / tpb);
    switch (N) {
    case 2: mrb_ref::both_kernel<2><<<grid, tpb>>>(B, barrier_default, dxi, xi, u_ref, it_ref, u_new, it_new); break;
    case 3: mrb_ref::both_kernel<3><<<grid, tpb>>>(B, barrier_default, dxi, xi, u_ref, it_ref, u_new, it_new); break;
    case 4: mrb_ref::both_kernel<4><<<grid, tpb>>>(B, barrier_default, dxi, xi, u_ref, it_ref, u_new, it_new); break;
    default: return (int)cudaErrorInvalidValue;
    }
    const cudaError_t st = cudaGetLastError();
    return st == cudaSuccess ? (int)cudaDeviceSynchronize() : (int)st;
}
