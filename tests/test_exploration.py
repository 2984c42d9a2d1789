"""Exploratory action selection (mrb_select_actions, csrc/explore.cu; policy.Exploration).

The random-number contract is exact (include/marbler_b200.h), so the kernel is compared with a numpy replica of it
draw for draw: a vectorised Philox4x32-10, pinned to the oracle's C Philox and the Random123 known answers, and the
two selection rules.  The one place where the replica can legitimately disagree is a softmax draw that lands within
rounding of a boundary of the cumulative sum (exp on the device and in numpy may differ in the last bit); those are
counted and must not occur at the sizes used here."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import golden_util as gu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASK = np.uint64(0xFFFFFFFF)
SEED = 0x0123456789ABCDEF
CANARY = -12345
MRB_E_ARG = -1


# ------------------------------------------------------------------------------------------------ the replica

def philox(c, k):
    """Philox4x32-10 over arrays: c = 4 counter words, k = 2 key words (anything uint32-valued) -> 4 uint64 arrays."""
    a0, a1, a2, a3 = (np.asarray(x, dtype=np.uint64) & MASK for x in c)
    k0, k1 = (np.asarray(x, dtype=np.uint64) & MASK for x in k)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * a0, np.uint64(0xCD9E8D57) * a2
        a0, a1, a2, a3 = (p1 >> np.uint64(32)) ^ a1 ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ a3 ^ k1, p0 & MASK
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK, (k1 + np.uint64(0xBB67AE85)) & MASK
    return a0, a1, a2, a3


def draws(seed, env_id0, B, N, t):
    """w0..w3 of every (env, agent) row at step t: counter (gid lo, gid hi, (uint32) t, 0x80000000 | agent)."""
    gid = np.uint64(env_id0) + np.repeat(np.arange(B, dtype=np.uint64), N)
    agent = np.tile(np.arange(N, dtype=np.uint64), B)
    t32 = np.full(B * N, t & 0xFFFFFFFF, dtype=np.uint64)
    return philox((gid & MASK, gid >> np.uint64(32), t32, np.uint64(0x80000000) | agent), (seed & 0xFFFFFFFF, seed >> 32))


def epsilon(t, eps_start, eps_finish, anneal_time):
    return max(eps_finish, eps_start - (eps_start - eps_finish) * t / anneal_time)


def epsilon_greedy(w, greedy, A, eps):
    """-> (actions, explored mask)"""
    thr = 2 ** 32 if eps >= 1.0 else int(np.floor(eps * 2.0 ** 32))
    explore = w[0] < np.uint64(thr)
    act = ((w[1] * np.uint64(A)) >> np.uint64(32)).astype(np.int32)
    return np.where(explore, act, greedy.reshape(-1)).astype(np.int32), explore


def softmax(w, q):
    """q [rows, A] float32 -> (actions, rows whose draw lies within 1e-12 S of a running-sum boundary)."""
    qd = q.astype(np.float64)
    e = np.exp(qd - q.max(axis=1).astype(np.float64)[:, None])
    c = np.add.accumulate(e, axis=1)                     # running sums in index order; the last one is S
    S = c[:, -1]
    u = ((w[2] >> np.uint64(5)).astype(np.float64) * 67108864.0 + (w[3] >> np.uint64(6)).astype(np.float64)) / 2.0 ** 53
    target = u * S
    over = c > target[:, None]
    last = e.shape[1] - 1 - np.argmax((e > 0)[:, ::-1], axis=1)
    act = np.where(over.any(axis=1), np.argmax(over, axis=1), last).astype(np.int32)
    near = (np.abs(c - target[:, None]) < 1e-12 * S[:, None]).any(axis=1)
    return act, near


# ------------------------------------------------------------------------------------------------ CPU tests

def test_replica_philox_is_the_oracles(oracle_lib):
    for ctr, key, want in (([0] * 4, [0] * 2, [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
                           ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
                           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
                            [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])):
        assert [int(v) for v in philox(ctr, key)] == want
    rng = np.random.RandomState(7)
    ctr = rng.randint(0, 2 ** 32, size=(4, 3000), dtype=np.uint64)
    key = rng.randint(0, 2 ** 32, size=(2, 3000), dtype=np.uint64)
    got = np.stack(philox(ctr, key))
    for i in range(3000):
        assert oracle_lib.philox([int(v) for v in ctr[:, i]], [int(v) for v in key[:, i]]) == [int(v) for v in got[:, i]], i


def test_select_actions_rejects_bad_arguments():
    from marbler_b200 import _lib, build
    build.build()
    lib = _lib.load()
    step = np.zeros(1, dtype=np.int64)
    q = np.zeros(64, dtype=np.float32)
    act = np.zeros(64, dtype=np.int32)
    P = lambda a: C.c_void_p(a.ctypes.data)

    def desc(**kw):
        d = _lib.SelectDesc(C.sizeof(_lib.SelectDesc), _lib.SELECT_EPSILON_GREEDY, 1, 0, 1.0, 0.05, 100)
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    def call(d=None, B=4, N=4, A=5, step_p=P(step), q_p=P(q), act_p=P(act), null_desc=False):
        d = desc() if d is None else d
        return lib.mrb_select_actions(0, B, N, A, None if null_desc else C.byref(d), step_p, q_p, act_p, None)

    cases = [
        (dict(null_desc=True), b"required"), (dict(step_p=None), b"required"), (dict(act_p=None), b"required"),
        (dict(d=desc(struct_size=8)), b"struct_size"), (dict(d=desc(mode=0)), b"unknown mode"),
        (dict(d=desc(mode=3)), b"unknown mode"), (dict(B=0), b">= 1"), (dict(N=0), b">= 1"), (dict(A=0), b">= 1"),
        (dict(B=2 ** 40), b"2^39"),
        (dict(d=desc(eps_start=-0.1)), b"[0, 1]"), (dict(d=desc(eps_start=1.5)), b"[0, 1]"),
        (dict(d=desc(eps_finish=-1e-9)), b"[0, 1]"), (dict(d=desc(eps_finish=float("nan"))), b"[0, 1]"),
        (dict(d=desc(anneal_time=0)), b"anneal_time"), (dict(d=desc(anneal_time=-5)), b"anneal_time"),
        (dict(d=desc(mode=_lib.SELECT_SOFTMAX), q_p=None), b"softmax needs q"),
    ]
    for kw, msg in cases:
        assert call(**kw) == MRB_E_ARG, kw
        assert msg in lib.mrb_last_error(None), (kw, lib.mrb_last_error(None))


# ------------------------------------------------------------------------------------------------ GPU tests

def _explore(mode, t=0, **kw):
    from marbler_b200.policy import Exploration
    ex = Exploration(mode, seed=kw.pop("seed", SEED), device="cuda:0", **kw)
    ex.step.fill_(t)
    return ex


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 63, 65, 65536])
def test_epsilon_greedy_is_the_replica(B):
    rng = np.random.RandomState(B)
    for N in (1, 4, 20, 32):
        rows = B * N
        for t in (0, 7, 2 ** 31 + 5):
            w = draws(SEED, 0, B, N, t)
            for A in (1, 2, 5, 20, 24):
                greedy = rng.randint(0, A, size=rows).astype(np.int32)
                buf = torch.full((rows + 64,), CANARY, dtype=torch.int32, device="cuda:0")
                actions = buf[:rows].view(B, N)
                q = torch.randn((B, N, A), device="cuda:0")
                q0 = q.clone()
                for eps in (0.0, 0.3, 1.0):
                    ex = _explore("epsilon_greedy", t, eps_start=eps, eps_finish=eps, anneal_time=1)
                    actions.copy_(torch.as_tensor(greedy.reshape(B, N)))
                    ex.select(actions, q)
                    got = buf.cpu().numpy()
                    want, explored = epsilon_greedy(w, greedy, A, eps)
                    case = (N, t, A, eps)
                    assert np.array_equal(got[:rows], want), case
                    assert (got[rows:] == CANARY).all(), case
                    assert int(ex.step.item()) == t + 1, case
                    if eps == 0.0:
                        assert not explored.any() and np.array_equal(got[:rows], greedy), case
                    if eps == 1.0:
                        assert explored.all(), case
                assert torch.equal(q, q0)


@pytest.mark.gpu
def test_schedule_and_counter():
    B, N, A, at = 4096, 4, 5, 1000
    greedy = np.full(B * N, -1, dtype=np.int32)                  # explored rows are the ones that change
    for t in (0, at // 2, at, 3 * at):
        ex = _explore("epsilon_greedy", t, eps_start=1.0, eps_finish=0.05, anneal_time=at)
        eps = epsilon(t, 1.0, 0.05, at)
        assert ex.epsilon() == eps
        actions = torch.as_tensor(greedy.reshape(B, N)).cuda()
        ex.select(actions, n_actions=A)
        got = actions.cpu().numpy().reshape(-1)
        want, explored = epsilon_greedy(draws(SEED, 0, B, N, t), greedy, A, eps)
        assert np.array_equal(got != -1, explored) and np.array_equal(got, want), t
        assert 0.0 < explored.mean() and (explored.mean() == 1.0) == (t == 0)
    # consecutive calls draw at t, t + 1, ... and leave the counter at start + calls
    start, calls = 41, 5
    ex = _explore("epsilon_greedy", start, eps_start=1.0, eps_finish=0.05, anneal_time=at)
    for k in range(calls):
        actions = torch.as_tensor(greedy.reshape(B, N)).cuda()
        ex.select(actions, n_actions=A)
        want, _ = epsilon_greedy(draws(SEED, 0, B, N, start + k), greedy, A, epsilon(start + k, 1.0, 0.05, at))
        assert np.array_equal(actions.cpu().numpy().reshape(-1), want), k
    assert int(ex.step.item()) == start + calls


def _softmax_case(q, t=3):
    B, N, A = q.shape
    ex = _explore("softmax", t)
    qd = torch.as_tensor(q).cuda()
    actions = torch.full((B, N), CANARY, dtype=torch.int32, device="cuda:0")
    ex.select(actions, qd)
    assert torch.equal(qd.cpu(), torch.as_tensor(q))
    want, near = softmax(draws(SEED, 0, B, N, t), q.reshape(B * N, A))
    got = actions.cpu().numpy().reshape(-1)
    assert int(near.sum()) == 0
    assert np.array_equal(got, want), int((got != want).sum())
    return got


@pytest.mark.gpu
def test_softmax_is_the_replica():
    rng = np.random.RandomState(11)
    B, N = 65536, 4
    q = (rng.standard_normal((B, N, 5)) * 3).astype(np.float32)
    q[:1000] = 0.5                                               # every logit tied
    q[1000:2000, :, 1] = q[1000:2000, :, 3] = 9.0                # two tied maxima
    q[2000:3000] = 0.0
    q[2000:3000, :, 2] = 100.0                                   # one logit 100 above the rest
    got = _softmax_case(q).reshape(B, N)
    assert (got[2000:3000] == 2).all()
    assert (_softmax_case(np.zeros((B, N, 1), dtype=np.float32)) == 0).all()
    _softmax_case((rng.standard_normal((B, N, 24)) * 2).astype(np.float32), t=2 ** 31 + 5)
    _softmax_case((rng.standard_normal((63, 20, 20))).astype(np.float32))
    # frequencies over 262,144 draws of one fixed distribution sit within 5 sigma of its probabilities
    logits = np.array([0.5, -1.0, 2.0, 0.0, 1.0], dtype=np.float32)
    got = _softmax_case(np.broadcast_to(logits, (B, N, 5)).copy(), t=9)
    p = np.exp(logits.astype(np.float64) - logits.max())
    p /= p.sum()
    n = B * N
    count = np.bincount(got, minlength=5)
    assert (np.abs(count - n * p) < 5 * np.sqrt(n * p * (1 - p))).all(), (count, n * p)


def _load_pcp():
    z = np.load(os.path.join(gu.GOLDEN, "policy", "PredatorCapturePrey_vdn.npz"))
    return {k[3:]: z[k] for k in z.files if k.startswith("sd.")}


KERNEL_NAME = {"tc2": "policy_act_tc2_kernel", "mma": "policy_act_kernel<", "f32": "policy_act_f32_kernel"}


def _kernel_run(accurate):
    """Greedy and epsilon-greedy actions of the shipped PredatorCapturePrey checkpoint on 4,096 envs, and the policy
    kernels the explored call launched."""
    from trace_util import kernels_launched
    from marbler_b200.policy import Policy
    B, N, D = 4096, 4, 16
    pol = Policy(_load_pcp(), N, D, device="cuda:0", accurate=accurate)
    g = torch.Generator(device="cuda:0").manual_seed(5)
    obs = torch.rand((B, N, D), generator=g, device="cuda:0") * 2 - 1
    hid = (torch.rand((B, N, 128), generator=g, device="cuda:0") - 0.5)
    greedy = pol.act(obs, hid.clone())
    ex = _explore("epsilon_greedy", 17, eps_start=0.3, eps_finish=0.3, anneal_time=1)
    out = {}
    names = kernels_launched(lambda: out.setdefault("a", pol.act(obs, hid.clone(), explore=ex)), "policy_act")
    return greedy.cpu().numpy(), out["a"].cpu().numpy(), names


def _dump_kernel_run(path, accurate):
    greedy, explored, names = _kernel_run(accurate)
    np.savez(path, greedy=greedy, explored=explored, names=np.array(names))


@pytest.mark.gpu
def test_exploration_is_independent_of_the_policy_kernel(tmp_path):
    """Each kernel runs in a subprocess: MRB_POLICY_TC is read once per process, and profiler sessions opened here in
    the test process were seen to leave the traces of later tests (test_policy_kernels.py) empty."""
    runs = {}
    for kernel, accurate, tc in (("tc2", False, "1"), ("mma", False, "0"), ("f32", True, "1")):
        path = str(tmp_path / (kernel + ".npz"))
        code = "import sys; sys.path[:0] = [%r, %r]; import test_exploration as t; t._dump_kernel_run(%r, %r)" % (
            ROOT, os.path.join(ROOT, "tests"), path, accurate)
        res = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, MRB_POLICY_TC=tc), capture_output=True,
                             text=True, timeout=600)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
        z = np.load(path)
        assert len(z["names"]) and all(KERNEL_NAME[kernel] in str(n) for n in z["names"]), (kernel, z["names"])
        runs[kernel] = (z["greedy"], z["explored"])
    B, N = runs["tc2"][0].shape
    w = draws(SEED, 0, B, N, 17)
    for kernel, (greedy, explored) in runs.items():
        want, mask = epsilon_greedy(w, greedy, 5, 0.3)
        assert np.array_equal(explored.reshape(-1), want), kernel
    mask = epsilon_greedy(w, runs["tc2"][0], 5, 0.3)[1]
    assert 0.25 < mask.mean() < 0.35
    ref = runs["f32"][1].reshape(-1)
    for kernel in ("tc2", "mma"):
        a = runs[kernel][1].reshape(-1)
        assert np.array_equal(a[mask], ref[mask]), kernel                       # explored rows: identical
        assert (a[~mask] == ref[~mask]).mean() > 0.99, kernel                   # exploited rows: near-ties may flip


@pytest.mark.gpu
def test_softmax_act_allocates_q():
    from marbler_b200.policy import Policy
    B, N, D = 1000, 4, 16
    pol = Policy(_load_pcp(), N, D, device="cuda:0")
    obs = torch.rand((B, N, D), generator=torch.Generator(device="cuda:0").manual_seed(2), device="cuda:0")
    q = torch.zeros((B, N, 5), device="cuda:0")
    a1 = pol.act(obs, pol.init_hidden(B), explore=_explore("softmax", 4))
    a2 = pol.act(obs, pol.init_hidden(B), q=q, explore=_explore("softmax", 4))
    want, near = softmax(draws(SEED, 0, B, N, 4), q.cpu().numpy().reshape(B * N, 5))
    assert torch.equal(a1, a2) and not near.any() and np.array_equal(a1.cpu().numpy().reshape(-1), want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["epsilon_greedy", "softmax"])
def test_sharded_halves_draw_what_one_batch_draws(mode):
    B, N, A = 4096, 4, 5
    rng = np.random.RandomState(3)
    greedy = torch.as_tensor(rng.randint(0, A, size=(B, N)).astype(np.int32)).cuda()
    q = torch.as_tensor(rng.standard_normal((B, N, A)).astype(np.float32)).cuda()
    whole = greedy.clone()
    _explore(mode, 23, env_id0=0, eps_start=0.3, eps_finish=0.3).select(whole, q, n_actions=A)
    halves = greedy.clone()
    for lo in (0, B // 2):
        part = halves[lo:lo + B // 2]                            # a contiguous view: the rank's own batch
        _explore(mode, 23, env_id0=lo, eps_start=0.3, eps_finish=0.3).select(part, q[lo:lo + B // 2], n_actions=A)
    assert torch.equal(whole, halves)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["epsilon_greedy", "softmax"])
def test_graph_replay_equals_eager(mode):
    from marbler_b200.policy import Policy, Rollout
    from marbler_b200.vec_env import VecEnv
    sd, cfg = _load_pcp(), dict(gu.Golden("PredatorCapturePrey_rollout").cfg)

    def make(use_graph):
        env = VecEnv("PredatorCapturePrey", cfg, num_envs=1024, device="cuda:0", seed=21, auto_reset=True)
        ex = _explore(mode, 0, eps_start=1.0, eps_finish=0.05, anneal_time=8)     # eps moves during the run
        return Rollout(env, Policy(sd, 4, 16, device="cuda:0"), use_graph=use_graph, steps_per_graph=4, explore=ex)
    r1, r2 = make(True), make(False)
    r1.reset(), r2.reset()
    r1.run(13), r2.run(13)
    torch.cuda.synchronize()
    assert r1._graph is not None
    assert torch.equal(r1.env.state_f64, r2.env.state_f64) and torch.equal(r1.env.state_i32, r2.env.state_i32)
    assert torch.equal(r1.hidden, r2.hidden) and torch.equal(r1.actions, r2.actions)
    assert torch.equal(r1.env.stats, r2.env.stats) and torch.equal(r1.env.obs, r2.env.obs)
    assert int(r1.explore.step.item()) == int(r2.explore.step.item()) == 13
    r1.reset()
    assert int(r1.explore.step.item()) == 13                    # reset does not rewind the schedule


@pytest.mark.gpu
def test_epsilon_greedy_rollout_follows_the_host_loop(oracle_lib):
    """The float32 policy plus epsilon-greedy (eps 0.2) in closed loop against the float32 torch agent, the replica's
    draws and the C oracle env: explored rows are exact at every step, and every env follows action for action."""
    from test_policy import _cpu_agent
    from marbler_b200.policy import Policy, Rollout
    from marbler_b200.vec_env import VecEnv
    sd, cfg = _load_pcp(), dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    B, T, N, D = 1024, 12, 4, 16
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=21, auto_reset=True)
    ex = _explore("epsilon_greedy", 0, seed=99, eps_start=0.2, eps_finish=0.2)
    ro = Rollout(env, Policy(sd, N, D, device="cuda:0", accurate=True), use_graph=False, explore=ex)
    ro.reset()
    orc = oracle_lib.COracle("PredatorCapturePrey", cfg)
    sf, si = orc.reset_flat(B, seed=21, threads=8)
    h = torch.zeros(B * N, 128)
    obs = np.zeros((B, N, D))
    fresh = np.ones(B, dtype=bool)
    follow = np.ones(B, dtype=bool)
    eye = torch.eye(N).repeat(B, 1)
    for t in range(T):
        ro.run(1)
        torch.cuda.synchronize()
        o = torch.tensor(obs, dtype=torch.float32)
        o[torch.tensor(fresh)] = 0
        h = h.reshape(B, N, 128)
        h[torch.tensor(fresh)] = 0
        q, h = _cpu_agent(sd, torch.cat([o.reshape(B * N, D), eye], dim=1), h.reshape(B * N, 128))
        greedy = q.argmax(dim=1).numpy().astype(np.int32)
        a, explored = epsilon_greedy(draws(99, 0, B, N, t), greedy, 5, 0.2)
        got = ro.actions.cpu().numpy().reshape(-1)
        assert np.array_equal(got[explored], a[explored]), t
        follow &= (got == a).reshape(B, N).all(axis=1)
        obs, rew, dist, out_i = orc.step_flat(sf, si, a.reshape(B, N), auto_reset=True, seed=21, threads=8)
        fresh = out_i[:, 1].astype(bool)
    assert follow.mean() >= 0.999, follow.mean()


@pytest.mark.gpu
def test_each_call_is_two_launches():
    from marbler_b200 import _lib
    lib = _lib.load()
    actions = torch.zeros((100, 4), dtype=torch.int32, device="cuda:0")
    q = torch.zeros((100, 4, 5), device="cuda:0")
    ex, sm = _explore("epsilon_greedy"), _explore("softmax")
    n0 = lib.mrb_launch_count()
    for _ in range(3):
        ex.select(actions, n_actions=5)
        sm.select(actions, q)
    assert lib.mrb_launch_count() - n0 == 12
