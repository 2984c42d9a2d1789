"""The N <= 4 barrier-QP iteration (QpDual<N>, LDL' factor) against the Cholesky iteration it replaced.

tests/qp_reference/qp_dual_cholesky.cu keeps the previous iteration verbatim and runs both on the same problems in one
kernel.  The rewrite changes rounding only (one reciprocal per pivot instead of an rsqrt, gap * (1/m) instead of gap / m),
so on every problem the iteration counts must be equal and the velocities equal to 1e-10 relative: on QPs taken from
running PredatorCapturePrey envs and on hard layouts (pairs inside the safety radius, where the barrier gain is 1e6,
and near-coincident robots)."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from qp_util import _hard_layouts

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = os.path.join(ROOT, "tests", "qp_reference", "qp_dual_cholesky.cu")
REL_TOL = 1e-10


@pytest.fixture(scope="module")
def ref_lib():
    from marbler_b200 import build as mb
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    tmp = tempfile.mkdtemp(prefix="qp_dual_ref_")
    so = os.path.join(tmp, "qp_dual_cholesky.so")
    flags = [f for f in mb.NVCC_FLAGS if f != "-lineinfo"]
    res = subprocess.run([nvcc] + flags + ["-I", mb.CSRC, "-o", so, REF_SRC], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    lib = C.CDLL(so)
    lib.qp_both.argtypes = [C.c_int, C.c_int, C.c_int64] + [C.c_void_p] * 6
    lib.qp_both.restype = C.c_int
    yield lib
    shutil.rmtree(tmp, ignore_errors=True)


def _both(lib, dxi, xi, default):
    """dxi, xi [B, 2, N] numpy -> (u_ref, it_ref, u_new, it_new), u as [B, 2, N]"""
    B, _, N = dxi.shape
    d = torch.tensor(np.ascontiguousarray(dxi.transpose(1, 2, 0)), dtype=torch.float64, device="cuda:0")
    x = torch.tensor(np.ascontiguousarray(xi.transpose(1, 2, 0)), dtype=torch.float64, device="cuda:0")
    u_ref, u_new = torch.empty_like(d), torch.empty_like(d)
    it_ref = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    it_new = torch.zeros_like(it_ref)
    torch.cuda.synchronize()
    st = lib.qp_both(N, int(default), B, d.data_ptr(), x.data_ptr(), u_ref.data_ptr(), it_ref.data_ptr(),
                     u_new.data_ptr(), it_new.data_ptr())
    assert st == 0, "CUDA error %d" % st
    out = lambda u: u.cpu().numpy().transpose(2, 0, 1)
    return out(u_ref), it_ref.cpu().numpy(), out(u_new), it_new.cpu().numpy()


def _pcp_layouts(rng, B, steps):
    """xi (the projected points the controller constrains) of running PredatorCapturePrey envs after each of `steps`
    random steps, with velocities towards random goals clipped like the si controller's"""
    from marbler_b200 import config
    from marbler_b200.vec_env import VecEnv
    cfg = config.load_yaml(config.default_config_path("PredatorCapturePrey"))
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
    env.reset()
    gen = torch.Generator(device="cuda:0").manual_seed(3)
    xis = []
    for _ in range(steps):
        env.step(torch.randint(0, env.n_actions, (B, env.N), generator=gen, device="cuda:0", dtype=torch.int32))
        p = env.agent_poses.cpu().numpy()                           # [B, 3, N]
        xis.append(np.stack([p[:, 0] + 0.05 * np.cos(p[:, 2]), p[:, 1] + 0.05 * np.sin(p[:, 2])], axis=1))
    xi = np.concatenate(xis)
    goal = xi + rng.uniform(-0.4, 0.4, xi.shape)
    dxi = goal - xi
    n = np.linalg.norm(dxi, axis=1, keepdims=True)
    dxi *= np.minimum(1.0, 0.15 / np.maximum(n, 1e-300))
    return dxi, xi, env.N


def _check(lib, dxi, xi, what):
    for default in (False, True):
        u_ref, it_ref, u_new, it_new = _both(lib, dxi, xi, default)
        B = len(it_ref)
        assert np.isfinite(u_new).all(), what
        differ = np.nonzero(it_ref != it_new)[0]
        assert differ.size == 0, (what, default, differ[:8], it_ref[differ[:8]], it_new[differ[:8]])
        scale = np.abs(u_ref).reshape(B, -1).max(axis=1)
        err = np.abs(u_new - u_ref).reshape(B, -1).max(axis=1)
        rel = err / np.maximum(scale, 1e-300)
        assert (err <= REL_TOL * scale).all(), (what, default, rel.max(), int(np.argmax(rel)))
        print("%s default=%s: %d QPs, mean iterations %.2f, max |du| / |u| %.2e" % (what, default, B, it_new.mean(), rel.max()))


def test_pcp_envs_and_hard_layouts_match_the_cholesky_iteration(ref_lib):
    rng = np.random.RandomState(17)
    dxi, xi, N = _pcp_layouts(rng, 4096, 4)
    assert len(xi) >= 16384 and N == 4
    _check(ref_lib, dxi, xi, "PCP envs")
    for n in (2, 3, 4):
        dxi, xi = _hard_layouts(rng, 16384, n)
        _check(ref_lib, dxi, xi, "hard layouts N=%d" % n)


def test_library_kernel_runs_the_tested_iteration(ref_lib):
    """mrb_barrier_qp (the library's own stand-alone kernel) gives the iteration counts of the new iteration above"""
    from marbler_b200.vec_env import barrier_qp
    rng = np.random.RandomState(23)
    for n in (2, 3, 4):
        dxi, xi = _hard_layouts(rng, 4096, n)
        _, _, u_new, it_new = _both(ref_lib, dxi, xi, False)
        u, it = barrier_qp(torch.tensor(dxi, device="cuda:0"), torch.tensor(xi, device="cuda:0"))
        assert np.array_equal(it.cpu().numpy(), it_new), n
        scale = np.abs(u_new).reshape(len(it_new), -1).max(axis=1)
        assert (np.abs(u.cpu().numpy() - u_new).reshape(len(it_new), -1).max(axis=1) <= REL_TOL * scale).all(), n
