"""mrb_barrier_qp against the float64 C oracle (orc_barrier_qp, itself pinned to the cvxopt restatement by
tests/test_qp_oracle_anchor.py) and against the exact optimum, for every team size from 1 to 32 and both barrier kinds.

The kernels it reaches, by team size N:
  * N = 2..4  QpDual<N>, one problem per thread, 64-thread CTAs;
  * N = 5, 6  QpThread<N> (the primal solver), one problem per thread, 256-thread CTAs with the shared store;
  * N >= 7    one problem per warp, 4 per CTA: the FP64 tensor-core kernel of size N rounded up to a multiple of four
              (folded when N is one, padded with phantom robots otherwise) and, with MRB_WARP_GENERIC=1, the run-time
              team size kernel.  Both are checked against the same oracle results.
  * N = 1     the warp kernel with no constraints: the clipped dxi after 0 iterations.

Problem sets per (N, kind): hard layouts (a pair inside the safety radius, near-coincident robots), spawn-grid symmetric
layouts (the source of cvxopt's limit cycles), layouts from running envs (every scenario at its shipped team size and
PredatorCapturePrey at 8, 13, 20, 29 and 32 robots) and the edges of the 0.2 m/s velocity clip.

Over the problems the oracle solves in < 25 iterations (the rest are cvxopt's limit cycles, DESIGN.md section 2):
  * the iteration count equals the oracle's; where it does not, it differs by exactly one and both answers pass
    cvxopt's acceptance test against the exact (Lawson-Hanson NNLS) optimum;
  * |du| / max|u| is within a bar for well-conditioned problems and within a looser one where a pair sits inside the
    safety radius (safe barrier gain 1e6).
Every problem must give finite u and at most 50 iterations, and a sample of the well-posed GPU answers must pass the
acceptance test against the NNLS optimum on its own, independent of either restatement of cvxopt.

Every bar is 4-8x the worst case measured on a B200 (DESIGN.md section 2)."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest
import torch

from qp_util import (_dxi_edge_layouts, _exact, _grid_layouts, _hard_layouts, _problem, accepted, oracle_qp,
                     pair_inside)

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SETTLED = 25                     # oracle solves of >= 25 iterations are cvxopt's limit cycles: not reproducible
# per kernel family: (least fraction of equal iteration counts, max |du| / max|u| well-conditioned, with a pair inside
# the safety radius).  Measured on a B200: equal iteration counts on every settled problem of every family;
# |du| / max|u| at most 4.2e-9 / 1.0e-8 (dual), 1.1e-9 / 8.3e-9 (primal), 4.0e-10 / 6.6e-11 (tensor-core),
# 4.4e-10 / 9.7e-11 (generic)
BARS = {"dual": (0.999, 2e-8, 5e-8), "primal": (0.999, 5e-9, 4e-8), "tensor-core": (0.999, 2e-9, 5e-10),
        "generic": (0.999, 2e-9, 5e-10)}
MRB_E_ARG = -1

# running envs whose layouts are solved, by team size
ENVS = {4: [("PredatorCapturePrey", {}), ("MaterialTransport", {}), ("ArcticTransport", {}), ("Simple", {})],
        6: [("Warehouse", {})],
        8: [("PredatorCapturePrey", dict(predator=4, capture=4, ROBOT_INIT_RIGHT_THRESH=0.1))],
        13: [("PredatorCapturePrey", dict(predator=7, capture=6, ROBOT_INIT_RIGHT_THRESH=0.1))],
        20: [("PredatorCapturePrey", dict(predator=10, capture=10, ROBOT_INIT_RIGHT_THRESH=0.1))],
        29: [("PredatorCapturePrey", dict(predator=15, capture=14, ROBOT_INIT_RIGHT_THRESH=0.1))],
        32: [("PredatorCapturePrey", dict(predator=16, capture=16, ROBOT_INIT_RIGHT_THRESH=0.4))]}


def _total(N):
    return 16384 if N <= 6 else 1024 if N <= 16 else 256


def _paths(N):
    """(family, MRB_WARP_GENERIC) of every kernel mrb_barrier_qp reaches for N robots"""
    if N <= 4 and N >= 2:
        return [("dual", False)]
    if N <= 6 and N >= 5:
        return [("primal", False)]
    return [("tensor-core", False), ("generic", True)]


def _cta(family):
    return {"dual": 64, "primal": 256}.get(family, 4)


def _env_layouts(rng, B, N):
    """xi (the projected points the si controller constrains) of running envs after random steps, velocities towards
    random goals clipped like the si controller's"""
    from marbler_b200 import config
    from marbler_b200.vec_env import VecEnv
    cases = ENVS[N]
    xis = []
    for scenario, overrides in cases:
        cfg = config.load_yaml(config.default_config_path(scenario))
        cfg.update(overrides)
        per = -(-B // len(cases))
        envs = min(per, 1024)
        env = VecEnv(scenario, cfg, num_envs=envs, device=DEV, seed=3, auto_reset=True)
        env.reset()
        gen = torch.Generator(device=DEV).manual_seed(3)
        got = 0
        while got < per:
            env.step(torch.randint(0, env.n_actions, (envs, N), generator=gen, device=DEV, dtype=torch.int32))
            p = env.agent_poses.cpu().numpy()
            xis.append(np.stack([p[:, 0] + 0.05 * np.cos(p[:, 2]), p[:, 1] + 0.05 * np.sin(p[:, 2])], axis=1))
            got += envs
    xi = np.concatenate(xis)[:B]
    dxi = rng.uniform(-0.4, 0.4, xi.shape)
    n = np.linalg.norm(dxi, axis=1, keepdims=True)
    dxi *= np.minimum(1.0, 0.15 / np.maximum(n, 1e-300))
    return dxi, xi


def _problems(N):
    """(dxi, xi) [B, 2, N] of every problem set for N robots, and the name of each problem's set"""
    rng = np.random.RandomState(1000 + N)
    B = _total(N)
    sets = [("grid", _grid_layouts, B // 4), ("dxi-edges", _dxi_edge_layouts, B // 4)]
    if N in ENVS:
        sets.append(("envs", _env_layouts, B // 4))
    sets.insert(0, ("hard", _hard_layouts, B - sum(s[2] for s in sets)))
    dxi, xi, names = [], [], []
    for name, make, n in sets:
        d, x = make(rng, n, N)
        dxi.append(d)
        xi.append(x)
        names += [name] * n
    return np.concatenate(dxi), np.concatenate(xi), np.array(names)


@contextlib.contextmanager
def _warp_generic(on):
    """MRB_WARP_GENERIC=1 (read at every launch) selects the run-time team size warp kernel for N >= 7"""
    old = os.environ.pop("MRB_WARP_GENERIC", None)
    if on:
        os.environ["MRB_WARP_GENERIC"] = "1"
    try:
        yield
    finally:
        os.environ.pop("MRB_WARP_GENERIC", None)
        if old is not None:
            os.environ["MRB_WARP_GENERIC"] = old


def _gpu(dxi, xi, default, generic):
    from marbler_b200.vec_env import barrier_qp
    with _warp_generic(generic):
        u, it = barrier_qp(torch.tensor(dxi, device=DEV), torch.tensor(xi, device=DEV), barrier_default=default)
        torch.cuda.synchronize()
    return u.cpu().numpy(), it.cpu().numpy()


def _flat(u):
    """[2, N] -> [2N] interleaved (x0, y0, x1, ...), the order of _problem's variables"""
    return u.reshape(-1, order="F")


def _well_posed(d, A, b, ue):
    """the NNLS optimum is reliable: feasible to 1e-7 of |b| and not a metres-per-second answer of a pair inside the
    safety radius (test_qp_crosscheck.py)"""
    return A.shape[0] == 0 or (((A @ ue - b) / (1.0 + np.abs(b))).max() <= 1e-7 and np.abs(ue).max() <= 5.0)


@pytest.mark.parametrize("N", range(2, 33))
def test_barrier_qp_matches_the_oracle(N):
    dxi, xi, names = _problems(N)
    B = len(names)
    rng = np.random.RandomState(N)
    failures = []
    for default in (False, True):
        uo, ito = oracle_qp(dxi, xi, default)
        inside = np.array([pair_inside(x, default) for x in xi])
        scale = np.maximum(np.abs(uo).reshape(B, -1).max(axis=1), 1e-300)
        settled = ito < SETTLED
        for family, generic in _paths(N):
            min_equal, bar_well, bar_inside = BARS[family]
            label = "N=%d %s %s%s" % (N, "default" if default else "safe", family,
                                       " padded" if family == "tensor-core" and N % 4 else "")
            ug, itg = _gpu(dxi, xi, default, generic)
            rel = np.abs(ug - uo).reshape(B, -1).max(axis=1) / scale
            equal = settled & (itg == ito)
            differ = np.nonzero(settled & (itg != ito))[0]
            well, ill = equal & ~inside, equal & inside
            q = np.percentile(rel[well], [50, 99]) if well.any() else (0.0, 0.0)
            # the answers that stop one iteration apart: both must be answers cvxopt accepts
            rejected = []
            for b in differ:
                d, A, h = _problem(dxi[b], xi[b], default)
                ue = _exact(d, A, h)
                if _well_posed(d, A, h, ue) and not (accepted(_flat(ug[b]), d, A, h, ue) and accepted(_flat(uo[b]), d, A, h, ue)):
                    rejected.append(int(b))
            # the GPU answer against the exact optimum on a sample of well-posed problems
            cand = np.nonzero(settled & ~inside)[0]
            sample = rng.choice(cand, min(len(cand), 256 if N <= 6 else 48 if N <= 16 else 24), replace=False)
            nnls_checked, nnls_bad = 0, []
            for b in sample:
                d, A, h = _problem(dxi[b], xi[b], default)
                ue = _exact(d, A, h)
                if _well_posed(d, A, h, ue):
                    nnls_checked += 1
                    if not accepted(_flat(ug[b]), d, A, h, ue):
                        nnls_bad.append(int(b))
            print("QPREF %s: %d problems, %d settled, equal iterations %.5f, differ %d (by > 1: %d, rejected %d), "
                  "|du|/|u| well-conditioned max %.2e p99 %.2e median %.2e (%d), pair inside max %.2e (%d), "
                  "NNLS-accepted %d/%d, iterations max %d, finite %s" % (
                      label, B, settled.sum(), equal.sum() / max(settled.sum(), 1), len(differ),
                      int((np.abs(itg[differ] - ito[differ]) != 1).sum()), len(rejected),
                      rel[well].max() if well.any() else 0.0, q[1], q[0], well.sum(),
                      rel[ill].max() if ill.any() else 0.0, ill.sum(), nnls_checked - len(nnls_bad), nnls_checked,
                      itg.max(), np.isfinite(ug).all()))
            if not np.isfinite(ug).all() or itg.max() > 50 or itg.min() < 0:
                failures.append((label, "non-finite u or iterations outside [0, 50]"))
            if (np.abs(itg[differ] - ito[differ]) != 1).any():
                failures.append((label, "iteration counts differ by more than one", differ[:8]))
            if rejected:
                failures.append((label, "answers one iteration apart that cvxopt would not accept", rejected[:8]))
            if equal.sum() < min_equal * settled.sum():
                failures.append((label, "equal iteration counts", equal.sum() / settled.sum()))
            if well.any() and rel[well].max() > bar_well:
                failures.append((label, "well-conditioned |du|", rel[well].max(), names[well][np.argmax(rel[well])]))
            if ill.any() and rel[ill].max() > bar_inside:
                failures.append((label, "pair-inside |du|", rel[ill].max()))
            if nnls_bad or nnls_checked < len(sample) // 2:
                failures.append((label, "GPU answers rejected against the NNLS optimum", nnls_bad[:8], nnls_checked))
    assert not failures, failures


def test_one_robot_returns_the_clipped_velocity():
    rng = np.random.RandomState(1)
    dxi, xi = _dxi_edge_layouts(rng, 4096, 1)
    for default in (False, True):
        uo, ito = oracle_qp(dxi, xi, default)
        assert (ito == 0).all()
        n = np.linalg.norm(dxi, axis=1, keepdims=True)
        assert np.abs(uo - dxi * np.where(n > 0.2, 0.2 / np.maximum(n, 1e-300), 1.0)).max() <= 1e-15
        for generic in (False, True):
            ug, itg = _gpu(dxi, xi, default, generic)
            assert (itg == 0).all()
            scale = np.maximum(np.abs(uo).reshape(len(itg), -1).max(axis=1), 1e-300)
            assert (np.abs(ug - uo).reshape(len(itg), -1).max(axis=1) <= 1e-15 * scale).all()


def _raw(N, default, dxi, xi, with_iters=True, guard=64):
    """mrb_barrier_qp through ctypes on [B, 2, N] problems with NaN / sentinel guards after the end of u and iters;
    returns (rc, u [B, 2, N], iters [B] or None, u guard, iters guard)"""
    from marbler_b200 import _lib
    lib = _lib.load()
    B = dxi.shape[0]
    d = torch.tensor(np.ascontiguousarray(dxi.transpose(1, 2, 0)), device=DEV)
    x = torch.tensor(np.ascontiguousarray(xi.transpose(1, 2, 0)), device=DEV)
    u = torch.full((2 * N * B + guard,), float("nan"), dtype=torch.float64, device=DEV)
    it = torch.full((B + guard,), -7, dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    rc = lib.mrb_barrier_qp(0, N, int(default), B, C.c_void_p(d.data_ptr()), C.c_void_p(x.data_ptr()),
                            C.c_void_p(u.data_ptr()), C.c_void_p(it.data_ptr()) if with_iters else None, None)
    torch.cuda.synchronize()
    u, it = u.cpu().numpy(), it.cpu().numpy()
    return rc, u[:2 * N * B].reshape(2, N, B).transpose(2, 0, 1), it[:B], u[2 * N * B:], it[B:]


# (N, MRB_WARP_GENERIC) covering each kernel: both dual sizes' extremes, both primal sizes, the warp kernels folded,
# padded and generic
LAUNCH_CASES = [(2, False), (4, False), (5, False), (6, False), (8, False), (29, False), (13, True)]


@pytest.mark.parametrize("N,generic", LAUNCH_CASES, ids=["N=%d%s" % (n, " generic" if g else "") for n, g in LAUNCH_CASES])
def test_launch_edges(N, generic):
    """Batch sizes at the CTA edges: each problem's answer is the one it gets in a batch of 4,097, bit for bit, nothing
    is written past the end of u and iters, and a NULL iters pointer changes nothing"""
    family = _paths(N)[-1 if generic else 0][0]
    cta = _cta(family)
    rng = np.random.RandomState(N)
    dxi, xi = _hard_layouts(rng, 4097, N)
    with _warp_generic(generic):
        rc, u_all, it_all, ug, ig = _raw(N, False, dxi, xi)
        assert rc == 0 and np.isnan(ug).all() and (ig == -7).all()
        assert np.isfinite(u_all).all() and (it_all >= 1).all() and (it_all <= 50).all()
        for B in (1, cta - 1, cta, cta + 1, 2 * cta + 1, 4097):
            rc, u, it, ug, ig = _raw(N, False, dxi[:B], xi[:B])
            assert rc == 0, B
            assert np.isnan(ug).all() and (ig == -7).all(), (N, B, "wrote past the end")
            assert np.array_equal(u, u_all[:B]) and np.array_equal(it, it_all[:B]), (N, B)
            rc, u0, it0, ug, ig = _raw(N, False, dxi[:B], xi[:B], with_iters=False)
            assert rc == 0 and (it0 == -7).all() and (ig == -7).all() and np.isnan(ug).all(), (N, B)
            assert np.array_equal(u0, u), (N, B, "iters = NULL")
    from marbler_b200 import _lib
    d = torch.zeros(2 * 33 * 16, dtype=torch.float64, device=DEV)
    it = torch.zeros(16, dtype=torch.int32, device=DEV)
    for bad_N, bad_B in ((0, 16), (33, 16), (N, 0)):
        rc = _lib.load().mrb_barrier_qp(0, bad_N, 0, bad_B, C.c_void_p(d.data_ptr()), C.c_void_p(d.data_ptr()),
                                        C.c_void_p(d.data_ptr()), C.c_void_p(it.data_ptr()), None)
        assert rc == MRB_E_ARG, (bad_N, bad_B, rc)


COINCIDENT_CASES = [(2, False), (3, False), (4, False), (5, False), (6, False), (8, False), (11, False), (11, True),
                    (29, False), (32, True)]


@pytest.mark.parametrize("N,generic", COINCIDENT_CASES, ids=["N=%d%s" % (n, " generic" if g else "") for n, g in COINCIDENT_CASES])
def test_exactly_coincident_robots_stay_bounded(N, generic):
    """Two (or three) robots at exactly the same point: the constraint row is zero and its bound negative, so the QP is
    infeasible.  What u should be there is not decided; the kernel must stay inside its rows and stop within 50
    iterations.  Whether u is finite is printed per kernel."""
    rng = np.random.RandomState(7 + N)
    B = 512
    dxi, xi = _hard_layouts(rng, B, N)
    for b in range(B):
        i, j = rng.choice(N, 2, replace=False)
        xi[b][:, j] = xi[b][:, i]
        if N >= 3 and b % 2:
            k = [r for r in range(N) if r not in (i, j)][0]
            xi[b][:, k] = xi[b][:, i]
    with _warp_generic(generic):
        for default in (False, True):
            rc, u, it, ug, ig = _raw(N, default, dxi, xi)
            assert rc == 0
            assert np.isnan(ug).all() and (ig == -7).all(), "wrote past the end"
            assert (it >= 0).all() and (it <= 50).all(), (it.min(), it.max())
            uo, ito = oracle_qp(dxi[:64], xi[:64], default)
            print("QPCOINCIDENT N=%d%s %s: finite u in %d / %d problems (oracle: %d / 64), iterations max %d" % (
                N, " generic" if generic else "", "default" if default else "safe",
                np.isfinite(u).reshape(B, -1).all(axis=1).sum(), B, np.isfinite(uo).reshape(64, -1).all(axis=1).sum(),
                it.max()))
