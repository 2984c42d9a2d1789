"""Which kernel mrb_step runs for a (scenario, team size) and mrb_barrier_qp for a team size, read from a profiler trace.
The parity tests pass whichever kernel did the work; this test pins the dispatch rules (csrc/kern_step_*.cu,
csrc/kern_misc.cu), restated here from DESIGN.md §4:
  * a team of N <= 6 robots steps on step_thread_kernel<SCN, N> (one env per thread);
  * N >= 7 steps on the kernel with the compile-time team size NC = N rounded up to a multiple of four,
    step_warp_kernel<SCN, team_ppl(NC), NC, team_warps(NC), N == NC>, if the scenario has one (TEAM_MAX);
  * any other N >= 7, and every N >= 7 under MRB_WARP_GENERIC=1, steps on the run-time team size kernel
    step_warp_kernel<SCN, PPL, 0, 4, true>, PPL = the pair slots per lane rounded up to 1, 2, 4, 6, 8 or 16;
  * mrb_barrier_qp runs qp_thread_kernel<N> for N = 2..6, qp_warp_kernel<team_ppl(NC), NC, N == NC> for N >= 7 and
    qp_warp_kernel<PPL, 0, true> for N = 1 and, for N >= 7, under MRB_WARP_GENERIC=1."""
import re

import numpy as np
import pytest
import torch

from test_gpu_parity import TEAM_CASES, TENSOR_TEAMS
from trace_util import kernels_launched

pytestmark = pytest.mark.gpu

SCENARIOS = ("PredatorCapturePrey", "Warehouse", "MaterialTransport", "ArcticTransport", "Simple")   # MRB_PCP ... MRB_SIMPLE
TEAM_MAX = {"PredatorCapturePrey": 32, "Warehouse": 12, "Simple": 16}     # largest compile-time team size per scenario


def team_ppl(n):
    return (n * (n - 1) // 2 + 31) // 32


def team_warps(n):
    """Warps per CTA of the compile-time team size kernels: as many as 227 KB of workspace hold, at most 20 / 16 / 12."""
    ws = ((2 * n * (n + 1) + 12 * n + 2 * n * (n | 1) + 1) & ~1) + 64 * ((n + 3) // 4)
    return min(227 * 1024 // (8 * ws), 20 if n <= 8 else 16 if n <= 16 else 12)


def runtime_ppl(n):
    return next(p for p in (1, 2, 4, 6, 8, 16) if team_ppl(n) <= p)


def expected_step(scenario, N, generic):
    scn = SCENARIOS.index(scenario)
    if N <= 6:
        return "step_thread_kernel", (scn, N)
    nc = (N + 3) // 4 * 4
    if not generic and nc <= TEAM_MAX.get(scenario, 0):
        return "step_warp_kernel", (scn, team_ppl(nc), nc, team_warps(nc), N == nc)
    return "step_warp_kernel", (scn, runtime_ppl(N), 0, 4, True)


def expected_qp(N, generic):
    if 2 <= N <= 6:
        return "qp_thread_kernel", (N,)
    nc = (N + 3) // 4 * 4
    if N >= 7 and not generic:
        return "qp_warp_kernel", (team_ppl(nc), nc, N == nc)
    return "qp_warp_kernel", (runtime_ppl(N), 0, True)


def _arg(t):
    t = t.strip()
    if t in ("true", "(bool)1"):
        return True
    if t in ("false", "(bool)0"):
        return False
    return int(t.replace("(int)", ""))


def launched(fn):
    """(kernel, template arguments) of the one library kernel `fn` launches."""
    names = kernels_launched(fn, "mrb::")
    assert len(names) == 1, names
    m = re.search(r"mrb::(\w+)<([^>]*)>", names[0])
    return m.group(1), tuple(_arg(a) for a in m.group(2).split(","))


STEP_CASES = ([(s, {}) for s in SCENARIOS] + TEAM_CASES + TENSOR_TEAMS + [
    ("PredatorCapturePrey", dict(predator=10, capture=10, ROBOT_INIT_RIGHT_THRESH=0.1, num_neighbors=3)),   # 20
    ("Warehouse", dict(n_agents=14, num_neighbors=3, start_dist=0.4)),                   # above Warehouse's largest
    ("Simple", dict(n_agents=17, ROBOT_INIT_RIGHT_THRESH=0.1)),                          # above Simple's largest
    ("MaterialTransport", dict(n_agents=7, n_fast_agents=4, n_slow_agents=3, start_dist=0.2)),
    ("MaterialTransport", dict(n_agents=8, n_fast_agents=4, n_slow_agents=4, start_dist=0.2))])


@pytest.mark.parametrize("generic", [False, True], ids=["default", "MRB_WARP_GENERIC"])
@pytest.mark.parametrize("scenario,overrides", STEP_CASES,
                         ids=["%s-%d" % (s, i) for i, (s, _) in enumerate(STEP_CASES)])
def test_step_kernel(monkeypatch, scenario, overrides, generic):
    from marbler_b200 import config
    from marbler_b200.vec_env import VecEnv
    if generic:
        monkeypatch.setenv("MRB_WARP_GENERIC", "1")
    cfg = config.load_yaml(config.default_config_path(scenario))
    cfg.update(overrides)
    env = VecEnv(scenario, cfg, num_envs=256, device="cuda:0", seed=3)
    env.reset()
    a = torch.as_tensor(np.random.RandomState(0).randint(0, env.n_actions, (env.B, env.N)), dtype=torch.int32, device=env.device)
    assert launched(lambda: env.step(a)) == expected_step(scenario, env.N, generic), (scenario, env.N)


@pytest.mark.parametrize("generic", [False, True], ids=["default", "MRB_WARP_GENERIC"])
def test_barrier_qp_kernel(monkeypatch, generic):
    from marbler_b200.vec_env import barrier_qp
    if generic:
        monkeypatch.setenv("MRB_WARP_GENERIC", "1")
    rng = np.random.RandomState(1)
    for N in range(1, 33):
        xi = torch.tensor(np.stack([rng.uniform(-1.5, 1.5, (64, N)), rng.uniform(-0.9, 0.9, (64, N))], axis=1), device="cuda:0")
        dxi = torch.tensor(rng.uniform(-0.3, 0.3, (64, 2, N)), device="cuda:0")
        assert launched(lambda: barrier_qp(dxi, xi)) == expected_qp(N, generic), N
