"""The C oracle's barrier QP (orc_barrier_qp) against the Python restatement of cvxopt's coneqp (oracle/shims/cvxopt)
with rps' options, at team sizes and on layouts the fixture vectors do not cover: pairs inside the safety radius,
near-coincident robots and spawn-grid symmetric layouts, for 2 to 13 robots and both barrier kinds.

The two restatements share no code, so where both stop before cvxopt's limit cycles (< 25 iterations) they must take
the same number of iterations and return the same velocities to rounding: 1e-9 relative, and 1e-6 where a pair sits
inside the safety radius (barrier gain 1e6; near-coincident robots make the answer 1e4 m/s and the KKT system nearly
singular).  This pins the float64 reference that
tests/test_barrier_qp_reference.py holds the CUDA kernels to."""
import os
import sys

import numpy as np
import pytest

from qp_util import FEASTOL, MAXITERS, RELTOL, _grid_layouts, _hard_layouts, _problem, oracle_qp, pair_inside

SHIMS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "shims")
REL_TOL = 1e-9                   # measured worst case 4.3e-12
REL_TOL_INSIDE = 1e-6            # a pair inside the safety radius (gain 1e6, |u| up to 1e4): measured worst case 9.2e-8


def _shim(d, A, b):
    if SHIMS not in sys.path:
        sys.path.insert(0, SHIMS)
    import cvxopt.solvers as cs
    r = cs.coneqp_l(2 * np.eye(d.size), -2 * d, A, b, dict(maxiters=MAXITERS, reltol=RELTOL, feastol=FEASTOL))
    return np.asarray(r["x"]).reshape(-1), r["iterations"]


@pytest.mark.parametrize("default", [False, True], ids=["safe", "default"])
@pytest.mark.parametrize("N", [2, 3, 4, 5, 6, 7, 9, 13])
def test_oracle_matches_the_cvxopt_restatement(oracle_lib, N, default):
    B = 96 if N <= 7 else 48
    rng = np.random.RandomState(100 * N + default)
    compared = 0
    for name, make in (("hard", _hard_layouts), ("grid", _grid_layouts)):
        dxi, xi = make(rng, B, N)
        u, it = oracle_qp(dxi, xi, default)
        for b in range(B):
            d, A, h = _problem(dxi[b], xi[b], default)
            us, its = _shim(d, A, h)
            if it[b] >= 25 or its >= 25:
                continue
            assert it[b] == its, (name, b, it[b], its)
            uo = u[b].reshape(-1, order="F")
            rel = np.abs(uo - us).max() / max(np.abs(us).max(), 1e-300)
            assert rel <= (REL_TOL_INSIDE if pair_inside(xi[b], default) else REL_TOL), (name, b, rel)
            compared += 1
    assert compared >= 1.8 * B, compared
