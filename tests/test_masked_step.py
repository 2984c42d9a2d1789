"""Masked env steps (mrb_step_masked, csrc/compact.cu and the list variants of the step kernels; VecEnv.step(active=),
Rollout(skip_finished=True)).

CPU: the symbol and ABI version, and the Python argument checks that need no device.  GPU: a masked step against a plain
step of a second env that starts every step from the same state (active envs bit for bit, inactive envs untouched),
over mask shapes, every step kernel family and enough steps for episodes to end and auto-reset; the stats counters; the
collections and evaluations of Rollout(skip_finished=True) against the same runs without it; the C argument checks."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from test_episode_batch import CHECKPOINTS, PCP20, _checkpoint, _random_agent

MRB_E_ARG, MRB_E_STATE = -1, -4
INT_STATS = ("episodes", "collisions", "boundary_exits", "scenario_metric", "env_steps", "qp_solves", "qp_iterations",
             "timeouts", "qp_stalls", "substeps")


@pytest.fixture(scope="module")
def lib():
    from marbler_b200 import _lib, build
    build.build()
    return _lib.load()


# ------------------------------------------------------------------------------------------------ CPU

def test_masked_step_symbol_and_abi_version(lib):
    from marbler_b200 import _lib
    raw = C.CDLL(_lib.LIB_PATH)
    assert "mrb_step_masked" in _lib.SYMBOLS and hasattr(raw, "mrb_step_masked")
    assert lib.mrb_version() == _lib.ABI_VERSION == 7


def test_masked_step_rejects_a_null_env(lib):
    assert lib.mrb_step_masked(None, C.c_void_p(4096), C.c_void_p(4096), None) == MRB_E_ARG


def test_active_mask_checks_need_no_device():
    from marbler_b200.vec_env import VecEnv
    env = VecEnv.__new__(VecEnv)                 # the fields active_mask reads, without a handle or a device
    env.B, env.device = 8, torch.device("cuda", 0)
    with pytest.raises(TypeError):
        env.active_mask(torch.ones(8, dtype=torch.int32))
    with pytest.raises(TypeError):
        env.active_mask(np.ones(8, dtype=np.uint8))
    with pytest.raises(ValueError, match="shape"):
        env.active_mask(torch.ones(7, dtype=torch.bool))
    with pytest.raises(ValueError, match="shape"):
        env.active_mask(torch.ones((8, 1), dtype=torch.uint8))
    with pytest.raises(ValueError, match="device"):
        env.active_mask(torch.ones(8, dtype=torch.bool))       # a host tensor


def test_skip_finished_needs_record_or_evaluate():
    from marbler_b200.policy import Rollout
    with pytest.raises(ValueError, match="skip_finished"):
        Rollout(None, None, skip_finished=True)


# ------------------------------------------------------------------------------------------------ GPU: one step

def _cfg(scenario, overrides):
    from marbler_b200 import config
    return dict(config.load_yaml(config.default_config_path(scenario)), **(overrides or {}))


def _env(scenario, B, overrides=None, seed=11, **kw):
    from marbler_b200.vec_env import VecEnv
    return VecEnv(scenario, _cfg(scenario, overrides), num_envs=B, device="cuda:0", seed=seed, auto_reset=True, **kw)


def _pcp(N):
    cfg = dict(predator=N // 2, capture=N - N // 2, num_neighbors=3)
    if N > 13:
        cfg.update(ROBOT_INIT_RIGHT_THRESH=0.1, start_dist=0.25 if N > 20 else 0.3)
    return cfg


# (scenario, overrides, B, MRB_WARP_GENERIC).  B is never a multiple of a CTA, so the last CTA is ragged; short
# episodes, so that episodes end and auto-reset within the steps of a test.
STEP_CASES = {
    "PCP": ("PredatorCapturePrey", {}, 1000, False),
    "Warehouse": ("Warehouse", {}, 1000, False),
    "MaterialTransport": ("MaterialTransport", {}, 1000, False),
    "ArcticTransport": ("ArcticTransport", {}, 1000, False),
    "Simple": ("Simple", {}, 1000, False),
    "PCP5": ("PredatorCapturePrey", dict(predator=3, capture=2, num_neighbors=4, capability_aware=True), 600, False),
    "PCP6": ("PredatorCapturePrey", _pcp(6), 600, False),
    "PCP8": ("PredatorCapturePrey", _pcp(8), 300, False),
    "PCP20": ("PredatorCapturePrey", PCP20, 300, False),
    "PCP29": ("PredatorCapturePrey", _pcp(29), 150, False),
    "PCP8-generic": ("PredatorCapturePrey", _pcp(8), 300, True),
    "PCP-robotarium": ("PredatorCapturePrey", dict(robotarium=True, update_frequency=10), 600, False),
}


def _masks(B, gen):
    """The mask shapes every step cycles through, as bool tensors [B]."""
    idx = torch.arange(B, device="cuda:0")
    single = torch.zeros(B, dtype=torch.bool, device="cuda:0")
    single[B // 3] = True
    return [torch.rand(B, generator=gen, device="cuda:0") < 0.5,
            torch.zeros(B, dtype=torch.bool, device="cuda:0"),
            torch.ones(B, dtype=torch.bool, device="cuda:0"),
            single,
            (idx // 32) % 2 == 1,                       # warp-aligned blocks
            idx >= B - 21,                              # the ragged last CTA only
            torch.rand(B, generator=gen, device="cuda:0") < 0.5]


OUTPUTS = ("obs", "reward", "done", "message", "remaining", "dist", "obs_f64", "reward_f64")


def _bits(t):
    """t as integers of its width: torch.equal on these is bit-for-bit equality."""
    return t.view({8: torch.int64, 4: torch.int32, 1: torch.uint8}[t.element_size()])


def _stats(env):
    from marbler_b200 import _lib
    return dict(zip(_lib.STAT_NAMES, env.stats.cpu().tolist()))


def _masked_against_plain(scenario, overrides, B, steps=28):
    """Env a steps masked, env b plain from a's state before every step; returns the number of active auto-resets."""
    ov = dict(overrides, max_episode_steps=6)
    a, b = (_env(scenario, B, ov, f64_outputs=True) for _ in range(2))
    a.reset(), b.reset()
    gen = torch.Generator(device="cuda:0").manual_seed(5)
    masks = _masks(B, gen)
    resets = 0
    active_steps = 0
    for t in range(steps):
        m = masks[t % len(masks)]
        b.state_f64.copy_(a.state_f64)
        b.state_i32.copy_(a.state_i32)
        before_f, before_i = a.state_f64.clone(), a.state_i32.clone()
        for name in OUTPUTS:
            getattr(a, name).view(torch.uint8).fill_(0xA5)          # canary in every byte of every output row
        actions = torch.randint(0, a.n_actions, (B, a.N), generator=gen, device="cuda:0", dtype=torch.int32)
        sa, sb = _stats(a), _stats(b)
        a.step(actions, active=m if t % 2 else m.to(torch.uint8))
        b.step(actions)
        torch.cuda.synchronize()
        da = {k: v - sa[k] for k, v in _stats(a).items()}
        db = {k: v - sb[k] for k, v in _stats(b).items()}
        n = int(m.sum())
        active_steps += n
        assert da["env_steps"] == n, (t, da["env_steps"], n)
        if n == B:
            assert all(da[k] == db[k] for k in INT_STATS), (t, da, db)
            assert da["return_sum"] == pytest.approx(db["return_sum"], rel=1e-12, abs=1e-9)
            assert da["length_sum"] == db["length_sum"]
        if n == 0:
            assert all(v == 0 for v in da.values()), da
        off = ~m
        for x, y, before in ((a.state_f64, b.state_f64, before_f), (a.state_i32, b.state_i32, before_i)):
            assert torch.equal(_bits(x[:, m]), _bits(y[:, m])), t
            assert torch.equal(_bits(x[:, off]), _bits(before[:, off])), t
        for name in OUTPUTS:
            x, y = getattr(a, name), getattr(b, name)
            assert torch.equal(_bits(x[m]), _bits(y[m])), (t, name)
            assert bool((x[off].flatten().view(torch.uint8) == 0xA5).all()), (t, name)
        resets += int((b.done.bool() & m).sum())
    assert _stats(a)["env_steps"] == active_steps
    return resets


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(STEP_CASES))
def test_masked_step_equals_plain_step_on_active_envs_and_leaves_the_others(case, monkeypatch):
    scenario, overrides, B, generic = STEP_CASES[case]
    if generic:
        monkeypatch.setenv("MRB_WARP_GENERIC", "1")
    assert _masked_against_plain(scenario, overrides, B) > 0           # episodes ended and auto-reset under the mask


# ------------------------------------------------------------------------------------------------ GPU: rollouts

def _explore(mode, seed=9):
    from marbler_b200.policy import Exploration
    return Exploration(mode, seed=seed, eps_start=0.3, eps_finish=0.05, anneal_time=50, device="cuda:0")


def _rollout(scenario, B, mode, skip, T=None, K=None, overrides=None, use_graph=True, env_id0=0, checkpoint=True):
    from marbler_b200.policy import EpisodeBatch, EvalLog, Policy, Rollout
    from marbler_b200.vec_env import VecEnv
    env = VecEnv(scenario, _cfg(scenario, overrides), num_envs=B, device="cuda:0", seed=21, env_id0=env_id0,
                 auto_reset=True)
    sd = _checkpoint(CHECKPOINTS[scenario]) if checkpoint and scenario in CHECKPOINTS else \
        _random_agent(env.N, env.D, env.n_actions)
    return Rollout(env, Policy(sd, env.N, env.D, device="cuda:0"), use_graph=use_graph, steps_per_graph=4,
                   explore=_explore(mode), record=EpisodeBatch(env, T) if T else None,
                   evaluate=EvalLog(env, K) if K else None, skip_finished=skip)


def _run(ro):
    """collect() and / or evaluate(), as the rollout has record / evaluate; the data of each and the env steps taken."""
    out = {}
    for name, fn, attr in (("collect", ro.collect, "record"), ("evaluate", ro.evaluate, "eval_log")):
        if getattr(ro, attr) is not None:
            ro.env.stats.zero_()
            data = fn()
            torch.cuda.synchronize()
            out[name] = ({k: v.clone() for k, v in data.items()}, _stats(ro.env)["env_steps"])
    return out


def _same_data(got, want):
    assert set(got) == set(want)
    for name in want:
        for f, v in want[name][0].items():
            assert torch.equal(_bits(got[name][0][f].contiguous()), _bits(v.contiguous())), (name, f)


def _check_pair(scenario, B, mode, T=None, K=None, overrides=None, checkpoint=True):
    plain = _rollout(scenario, B, mode, False, T, K, overrides, checkpoint=checkpoint)
    skip = _rollout(scenario, B, mode, True, T, K, overrides, checkpoint=checkpoint)
    want, got = _run(plain), _run(skip)
    _same_data(got, want)
    assert int(skip.explore.step.item()) == int(plain.explore.step.item())
    if "collect" in got and K is None:
        filled = int(got["collect"][0]["filled"].sum())
        assert got["collect"][1] == filled - B, (got["collect"][1], filled)
    if "evaluate" in got:
        assert bool((got["evaluate"][0]["count"] == K).all())
        assert got["evaluate"][1] < want["evaluate"][1]
    return got, want


@pytest.mark.gpu
def test_skip_finished_pcp_vdn_65536_epsilon_greedy():
    """The shipped PredatorCapturePrey vdn checkpoint at 65,536 envs: a collect() of 81 steps and an evaluate() of
    K = 3 episodes per env give the same data bit for bit with and without skip_finished."""
    _check_pair("PredatorCapturePrey", 65536, "epsilon_greedy", T=81)
    _check_pair("PredatorCapturePrey", 65536, "epsilon_greedy", K=3)


@pytest.mark.gpu
def test_skip_finished_arctic_qmix_ns_and_material_mappo_ns_softmax():
    _check_pair("ArcticTransport", 4096, "epsilon_greedy", T=40)
    _check_pair("ArcticTransport", 4096, "epsilon_greedy", K=2)
    _check_pair("MaterialTransport", 4096, "softmax", T=40)
    _check_pair("MaterialTransport", 4096, "softmax", K=2)


@pytest.mark.gpu
def test_skip_finished_on_the_20_robot_team_kernel():
    _check_pair("PredatorCapturePrey", 4096, "epsilon_greedy", T=40, overrides=PCP20, checkpoint=False)
    _check_pair("PredatorCapturePrey", 4096, "epsilon_greedy", K=1, overrides=PCP20, checkpoint=False)


@pytest.mark.gpu
def test_skip_finished_with_record_and_evaluate_together():
    """One rollout with both: collect() and evaluate() each equal the run without skip_finished."""
    _check_pair("PredatorCapturePrey", 4096, "epsilon_greedy", T=30, K=2)


@pytest.mark.gpu
def test_skip_finished_graph_replay_equals_eager_and_shards_equal_one_batch():
    B, T, K = 2048, 50, 2
    g = _rollout("PredatorCapturePrey", B, "epsilon_greedy", True, T, K)
    e = _rollout("PredatorCapturePrey", B, "epsilon_greedy", True, T, K, use_graph=False)
    for _ in range(2):
        got, want = _run(g), _run(e)
        _same_data(got, want)
        assert got["collect"][1] == want["collect"][1] and got["evaluate"][1] == want["evaluate"][1]
    assert g._graph is not None
    assert torch.equal(g.env.state_f64, e.env.state_f64) and torch.equal(g.env.state_i32, e.env.state_i32)
    halves = [_rollout("PredatorCapturePrey", B // 2, "epsilon_greedy", True, T, K, env_id0=lo) for lo in (0, B // 2)]
    whole = _run(_rollout("PredatorCapturePrey", B, "epsilon_greedy", True, T, K))
    parts = [_run(h) for h in halves]
    for name in whole:
        for f, v in whole[name][0].items():
            assert torch.equal(v, torch.cat([p[name][0][f] for p in parts])), (name, f)
        assert whole[name][1] == sum(p[name][1] for p in parts)


# ------------------------------------------------------------------------------------------------ GPU: arguments

@pytest.mark.gpu
def test_masked_step_checks_its_arguments():
    """A host, pinned-host or other-device mask, NULL or misaligned actions give MRB_E_ARG, an unbound env MRB_E_STATE,
    all without a launch and without touching the env; a good call is two launches."""
    from marbler_b200 import _lib
    env = _env("PredatorCapturePrey", 64)
    lib = env.lib
    env.reset()
    actions = torch.zeros((64, env.N), dtype=torch.int32, device="cuda:0")
    env.step(actions)
    torch.cuda.synchronize()
    before = [t.clone() for t in (env.state_f64, env.state_i32, env.obs, env.reward, env.done, env.stats)]
    good = torch.ones(64, dtype=torch.uint8, device="cuda:0")
    host = torch.ones(64, dtype=torch.uint8)
    pinned = torch.ones(64, dtype=torch.uint8).pin_memory()
    P = lambda t: C.c_void_p(t.data_ptr())
    n0 = lib.mrb_launch_count()
    for mask in (host, pinned):
        assert lib.mrb_step_masked(env.handle, P(actions), P(mask), None) == MRB_E_ARG
        assert b"device memory" in lib.mrb_last_error(env.handle) or b"active" in lib.mrb_last_error(env.handle)
    if torch.cuda.device_count() > 1:
        other = torch.ones(64, dtype=torch.uint8, device="cuda:1")
        assert lib.mrb_step_masked(env.handle, P(actions), P(other), None) == MRB_E_ARG
    assert lib.mrb_step_masked(env.handle, None, P(good), None) == MRB_E_ARG
    assert lib.mrb_step_masked(env.handle, C.c_void_p(actions.data_ptr() + 4), P(good), None) == MRB_E_ARG
    assert lib.mrb_step_masked(None, P(actions), P(good), None) == MRB_E_ARG
    h = C.c_void_p()
    _lib.check(lib.mrb_create(C.byref(env.c), 0, 64, 0, C.byref(h)))
    assert lib.mrb_step_masked(h, P(actions), P(good), None) == MRB_E_STATE and b"mrb_bind" in lib.mrb_last_error(h)
    lib.mrb_destroy(h)
    assert lib.mrb_launch_count() == n0
    torch.cuda.synchronize()
    after = (env.state_f64, env.state_i32, env.obs, env.reward, env.done, env.stats)
    assert all(torch.equal(x, y) for x, y in zip(before, after))
    with pytest.raises(ValueError):
        env.step(actions, active=host.bool())
    with pytest.raises(ValueError):
        env.step(actions, active=good[:63])
    assert lib.mrb_launch_count() == n0
    env.step(actions, active=good)
    assert lib.mrb_launch_count() == n0 + 2
