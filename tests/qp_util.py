"""Barrier-QP helpers shared by the QP tests: the problem rps builds, its exact optimum, layouts where solvers go wrong,
and the C oracle over a batch of problems.

Layout convention: dxi, xi and u are [B, 2, N] (row 0 holds the x components, row 1 the y components), as
`marbler_b200.vec_env.barrier_qp` takes and returns them."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
from scipy.optimize import nnls

FEASTOL = RELTOL = 1e-2          # the cvxopt options rps sets at import
ABSTOL = 1e-7                    # cvxopt's default, which rps keeps
MAXITERS = 50


def _problem(dxi, xi, default):
    """rps create_single_integrator_barrier_certificate{,2} (SURVEY App. A.8): min |u - dxi|^2  s.t.  A u <= b."""
    N = dxi.shape[1]
    dxi = dxi.copy()
    nrm = np.linalg.norm(dxi, axis=0)
    big = nrm > 0.2
    dxi[:, big] *= 0.2 / nrm[big]
    r2 = 0.17 ** 2 if default else 0.2 ** 2
    rows, b = [], []
    for i in range(N - 1):
        for j in range(i + 1, N):
            e = xi[:, i] - xi[:, j]
            h = e @ e - r2
            a = np.zeros(2 * N)
            a[2 * i:2 * i + 2], a[2 * j:2 * j + 2] = -2 * e, 2 * e
            rows.append(a)
            b.append((100.0 if (default or h >= 0) else 1e6) * h ** 3)
    return dxi.reshape(-1, order="F"), np.array(rows).reshape(-1, 2 * N), np.array(b)


def _exact(d, A, b):
    """Least-distance problem by Lawson-Hanson: min |u - d|  s.t.  A u <= b   <=>   NNLS on the dual."""
    # u = d - A' lam / 1 with lam >= 0 minimising |A' lam - ... |: solve  min_{lam>=0} |[A'; (b - A d)'] lam + [0; 1]|  (LDP)
    c = b - A @ d                                   # constraints in shifted variable y = u - d:  A y <= c
    E = np.vstack([-A.T, -c[None, :]])
    f = np.zeros(E.shape[0])
    f[-1] = 1.0
    lam, _ = nnls(E, f, maxiter=20 * E.shape[1] + 1000)
    r = E @ lam - f
    if abs(r[-1]) < 1e-14:                          # y = 0 is optimal only when d itself is feasible
        return d.copy()
    y = -r[:-1] / r[-1]
    return d + y


def accepted(u, d, A, b, ue):
    """cvxopt's acceptance test for an answer u [2N] (interleaved like d) of the problem (d, A, b) with exact optimum ue:
    primal feasibility max(A u - b) <= feastol * max(1, |b|), and an objective no more than the duality gap cvxopt
    stops at above the optimum's: reltol * |pcost| (pcost = f(u) - d'd) or abstol, whichever is larger.  An objective
    below the optimum's is the feastol infeasibility the first test bounds."""
    if A.shape[0] == 0:
        return np.allclose(u, d, rtol=0, atol=1e-15)
    if (A @ u - b).max() > FEASTOL * max(1.0, np.linalg.norm(b)):
        return False
    f = lambda x: float((x - d) @ (x - d))
    return f(u) - f(ue) <= max(RELTOL * abs(f(u) - d @ d), ABSTOL)


def pair_inside(xi, default):
    """Whether two robots of the layout xi [2, N] sit inside the safety radius (0.17 m for rps' default barrier, 0.2 m
    for the safe one): the safe barrier's gain is then 1e6 and the problem ill-conditioned."""
    N = xi.shape[1]
    if N < 2:
        return False
    e = xi[:, :, None] - xi[:, None, :]
    d2 = (e * e).sum(axis=0)[np.triu_indices(N, 1)]
    return bool((d2 < (0.17 ** 2 if default else 0.2 ** 2)).any())


def _hard_layouts(rng, B, N):
    xi = np.stack([rng.uniform(-1.5, 1.5, (B, N)), rng.uniform(-0.9, 0.9, (B, N))], axis=1)
    for b in range(B):
        k = b % 3
        if k == 0:                                   # a pair inside the safety radius (0.17 / 0.2)
            i, j = rng.choice(N, 2, replace=False)
            xi[b][:, j] = xi[b][:, i] + rng.uniform(-0.14, 0.14, 2)
        elif k == 1:                                 # near-coincident robots
            i, j = rng.choice(N, 2, replace=False)
            xi[b][:, j] = xi[b][:, i] + rng.uniform(-1e-3, 1e-3, 2)
    dxi = rng.uniform(-0.3, 0.3, (B, 2, N))
    return dxi, xi


def _grid_layouts(rng, B, N):
    """Robots on cells of an rps spawn grid (spacing 0.3 m, a single column included), the mirror-symmetric layouts on
    which cvxopt's iteration can fall into its limit cycle.  Velocities: towards one common goal (mirror-symmetric
    problem), all equal, or towards the mirror image of the layout; clipped to 0.15 m/s like the si controller's."""
    xi = np.empty((B, 2, N))
    dxi = np.empty((B, 2, N))
    for b in range(B):
        cols = 1 if b % 4 == 0 else int(rng.randint(1, 7))
        rows = max(6, -(-(N + 1) // cols))
        cells = rng.choice(cols * rows, N, replace=False) if b % 2 else np.arange(N)
        xi[b, 0] = -1.3 + 0.3 * (cells // rows)
        xi[b, 1] = -0.9 + 0.3 * (cells % rows)
        kind = b % 3
        if kind == 0:
            goal = np.array([[rng.uniform(-1, 1)], [xi[b, 1].mean()]])
        elif kind == 1:
            goal = xi[b] + np.array([[0.3], [0.0]])
        else:
            goal = np.stack([-xi[b, 0], xi[b, 1][::-1]])
        g = goal - xi[b]
        n = np.linalg.norm(g, axis=0)
        dxi[b] = g * np.minimum(1.0, 0.15 / np.maximum(n, 1e-300))
    return dxi, xi


def _dxi_edge_layouts(rng, B, N):
    """Random layouts (a third with a close pair) with the velocity edges of rps' 0.2 m/s magnitude limit: zero
    velocity, norms of exactly 0.2 (not clipped), norms above 0.2 (clipped), and one robot still among moving ones."""
    xi = np.stack([rng.uniform(-1.5, 1.5, (B, N)), rng.uniform(-0.9, 0.9, (B, N))], axis=1)
    for b in range(0, B, 3):
        if N >= 2:
            i, j = rng.choice(N, 2, replace=False)
            xi[b][:, j] = xi[b][:, i] + rng.uniform(-0.15, 0.15, 2)
    dxi = np.empty((B, 2, N))
    for b in range(B):
        kind = b % 4
        if kind == 0:
            dxi[b] = 0.0
        elif kind == 1:                              # |dxi| == 0.2 exactly: axis directions and a 3-4-5 triangle
            axis = rng.randint(0, 6, N)
            dxi[b] = np.array([[0.2, -0.2, 0.0, 0.0, 0.12, -0.16], [0.0, 0.0, 0.2, -0.2, 0.16, 0.12]])[:, axis]
        elif kind == 2:
            t = rng.uniform(0, 2 * np.pi, N)
            dxi[b] = np.stack([np.cos(t), np.sin(t)]) * rng.uniform(0.2, 5.0, N)
        else:
            dxi[b] = rng.uniform(-0.3, 0.3, (2, N))
            dxi[b][:, rng.randint(N)] = 0.0
    return dxi, xi


def oracle_qp(dxi, xi, default, threads=None):
    """The C oracle's orc_barrier_qp on every problem of [B, 2, N] arrays -> (u [B, 2, N], iters [B]).  Per-problem
    calls fan out over a thread pool: ctypes releases the GIL and the oracle's workspace is thread-local."""
    import c_oracle
    L = c_oracle.lib()
    dxi = np.ascontiguousarray(dxi, dtype=np.float64)
    xi = np.ascontiguousarray(xi, dtype=np.float64)
    B, _, N = dxi.shape
    u = np.empty_like(dxi)
    it = np.empty(B, dtype=np.int32)
    dp = C.POINTER(C.c_double)

    def run(lo, hi):
        for b in range(lo, hi):
            it[b] = L.orc_barrier_qp(N, int(default), dxi[b].ctypes.data_as(dp), xi[b].ctypes.data_as(dp),
                                     u[b].ctypes.data_as(dp))

    threads = max(1, min(threads or os.cpu_count() or 1, B))
    chunk = max(1, min(64, -(-B // threads)))
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda lo: run(lo, min(B, lo + chunk)), range(0, B, chunk)))
    return u, it
