"""Independent cross-checks of the barrier-QP oracle (SURVEY.md section 8c "cross-checks available without the real
deps").  rps and cvxopt cannot be installed, so the restated interior-point method (oracle/shims/cvxopt, and the C
restatement that is pinned to it) is checked against mathematics instead:

  (i)   the returned iterate satisfies the barrier constraints  A u <= b  to the primal-feasibility tolerance rps
        asks of cvxopt:  max(A u - b) <= feastol * max(1, |b|)  with feastol = 1e-2 (cvxopt stops on |rz| / resz0);
  (ii)  its objective is within reltol = 1e-2 (relative, plus the feasibility slack) of the EXACT optimum, computed
        by an unrelated algorithm (Lawson-Hanson least-distance programming on scipy's NNLS);
  (iii) the same restated IPM run with tight tolerances converges to that exact optimum (<= 1e-6), i.e. the
        iteration itself is a correct QP solver and the loose answers differ from it only by early stopping.
"""
import os
import sys

import numpy as np
import pytest

import golden_util as gu
from qp_util import _exact, _problem

SHIMS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "shims")


@pytest.mark.parametrize("N", sorted(gu.qp_vectors().keys()))
def test_qp_iterates_are_feasible_and_near_optimal(oracle_lib, N):
    v = gu.qp_vectors()[N]
    if SHIMS not in sys.path:
        sys.path.insert(0, SHIMS)
    import cvxopt.solvers as cs
    worst_gap = worst_tight = 0.0
    gaps = []
    for i in range(min(48, v["dxi"].shape[0])):
        default = bool(v["default"][i])
        d, A, b = _problem(v["dxi"][i], v["xi"][i], default)
        scale = 1.0 + np.abs(b)
        u = v["u"][i].reshape(-1, order="F")
        if v["iters"][i] < 50:                       # (i) feasible to cvxopt's own criterion
            assert (A @ u - b).max() <= 1e-2 * max(1.0, np.linalg.norm(b)), (N, i, (A @ u - b).max())
        ue = _exact(d, A, b)
        if ((A @ ue - b) / scale).max() > 1e-7 or np.abs(ue).max() > 5.0 or v["iters"][i] >= 50:
            continue    # robots already inside the safety radius (gain 1e6): near-infeasible, metres-per-second "solutions";
                        # cvxopt itself gives up there (status unknown at 50 iterations) and NNLS is not reliable either
        f = lambda x: float((x - d) @ (x - d))
        if v["iters"][i] < 50:                       # (ii) objective within reltol of the optimum (cvxopt: gap <= reltol * |cost|)
            cost = abs(f(u) - d @ d)                 # cvxopt's pcost = x'x - 2 d'x = f - d'd
            gaps.append((abs(f(u) - f(ue)), cost, np.abs(u - ue).max()))
            worst_gap = max(worst_gap, abs(f(u) - f(ue)))
        # (iii) the restated IPM with tight tolerances reaches the exact optimum
        r = cs.coneqp_l(2 * np.eye(d.size), -2 * d, A, b, dict(maxiters=100, abstol=1e-12, reltol=1e-11, feastol=1e-11))
        ut = np.asarray(r["x"]).reshape(-1)
        worst_tight = max(worst_tight, np.abs(ut - ue).max())
        assert np.abs(ut - ue).max() < 2e-6, (N, i, np.abs(ut - ue).max())
    assert worst_tight < 2e-6
    assert len(gaps) >= 8      # N = 20 fixtures are mostly crowded (many pairs inside the safety radius): fewer well-posed cases
    # measured: relative objective gap 2.3e-3 ... 7.4e-3 over the team sizes - the early stop rps configures, no more
    assert max(g[0] / max(g[1], 1e-9) for g in gaps) <= 1.2e-2
