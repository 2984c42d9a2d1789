"""Evaluation on the device (mrb_eval_begin / mrb_eval_step, csrc/eval.cu; policy.EvalLog, Rollout(evaluate=)).

CPU: the ABI (symbols, struct layout, version) and EvalLog's summary over hand-made tables, also gathered over two
gloo ranks.  GPU: the table against a float64 torch restatement of the accumulator rules after every env step, against
the env's own episode statistics, graph against eager, two shards against one batch, the first episode of every env
against a recorded EpisodeBatch, and the argument checks."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from test_episode_batch import CHECKPOINTS, PCP20, _checkpoint, _random_agent

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MRB_E_ARG, MRB_E_STATE = -1, -4
FIELDS = ("return", "length", "message", "timeout", "remaining", "dist")


@pytest.fixture(scope="module")
def lib():
    from marbler_b200 import _lib, build
    build.build()
    return _lib.load()


# ------------------------------------------------------------------------------------------------ CPU: ABI

def test_eval_symbols_are_exported_and_the_abi_version_moved_on(lib):
    from marbler_b200 import _lib
    raw = C.CDLL(_lib.LIB_PATH)
    for s in ("mrb_eval_begin", "mrb_eval_step"):
        assert s in _lib.SYMBOLS and hasattr(raw, s), s
    assert lib.mrb_version() == _lib.ABI_VERSION >= 6      # 5 added mrb_policy_load; mrb_eval_* came after it


def test_eval_table_struct_matches_the_header(tmp_path):
    """sizeof and every field offset of mrb_eval_table as a C compiler lays out the header, against the ctypes struct."""
    from marbler_b200 import _lib
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    names = [n for n, _ in _lib.EvalTableDesc._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "marbler_b200.h"\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(mrb_eval_table));\n' +
                   "".join('  printf("%%zu\\n", offsetof(mrb_eval_table, %s));\n' % n for n in names) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.EvalTableDesc)
    assert out[1:] == [getattr(_lib.EvalTableDesc, n).offset for n in names]


def test_eval_calls_reject_a_null_env(lib):
    from marbler_b200 import _lib
    d = _lib.EvalTableDesc(C.sizeof(_lib.EvalTableDesc), 3, *([4096] * 10))
    assert lib.mrb_eval_begin(None, C.byref(d), None) == MRB_E_ARG and b"env is NULL" in lib.mrb_last_error(None)
    assert lib.mrb_eval_step(None, C.byref(d), None) == MRB_E_ARG


# ------------------------------------------------------------------------------------------------ CPU: summary

def _table(rows_per_env, K):
    """A hand-made table: rows_per_env[b] = list of (return, length, message, timeout, remaining, dist); the rows
    past count hold garbage that the summary must not read."""
    B = len(rows_per_env)
    dt = {"return": torch.float64, "length": torch.int32, "message": torch.uint8, "timeout": torch.uint8,
          "remaining": torch.int32, "dist": torch.float32}
    t = {f: torch.full((B, K), 77, dtype=dt[f]) for f in FIELDS}
    for b, rows in enumerate(rows_per_env):
        for k, row in enumerate(rows):
            for f, v in zip(FIELDS, row):
                t[f][b, k] = v
    t["count"] = torch.tensor([len(r) for r in rows_per_env], dtype=torch.int32)
    return t


# 3 envs, K = 3; env 1 logged only one episode (count < K), env 2 none
ROWS = [[(-1.0, 10, 0, 0, 2, 1.5), (4.0, 81, 0, 1, 0, 3.0), (2.0, 5, 1, 0, 1, 0.5)],
        [(-7.0, 3, 3, 0, 2, 0.25)],
        []]


def test_summary_of_a_hand_made_table():
    from marbler_b200.policy import summarize_episodes
    s = summarize_episodes(_table(ROWS, 3), n_agents=4)
    r = np.array([-1.0, 4.0, 2.0, -7.0])
    assert s["episodes"] == 4
    assert s["return_mean"] == s["test_return_mean"] == -0.5
    assert s["return_std"] == s["test_return_std"] == pytest.approx(np.sqrt(np.mean((r + 0.5) ** 2)), rel=1e-15)
    assert s["return_sem"] == pytest.approx(np.sqrt(np.sum((r + 0.5) ** 2) / 3) / 2, rel=1e-15)
    # linear interpolation over the sorted returns -7, -1, 2, 4 at positions q * 3
    assert s["return_quantiles"] == pytest.approx({5: -7 + 0.15 * 6, 25: -7 + 0.75 * 6, 50: 0.5, 75: 2 + 0.25 * 2,
                                                   95: 2 + 0.85 * 2}, rel=1e-14)
    assert s["length_mean"] == s["test_ep_length_mean"] == (10 + 81 + 5 + 3) / 4
    assert s["collision_rate"] == 0.5 and s["boundary_rate"] == 0.25 and s["timeout_rate"] == 0.25
    assert s["remaining_mean"] == 1.25 and s["dist_mean"] == (1.5 + 3.0 + 0.5 + 0.25) / 4


def test_summary_per_agent_divides_the_returns_only():
    from marbler_b200.policy import summarize_episodes
    whole, per = summarize_episodes(_table(ROWS, 3), 4), summarize_episodes(_table(ROWS, 3), 4, per_agent=True)
    for k in ("return_mean", "return_std", "return_sem", "test_return_mean", "test_return_std"):
        assert per[k] == pytest.approx(whole[k] / 4, rel=1e-15), k
    assert per["return_quantiles"] == pytest.approx({q: v / 4 for q, v in whole["return_quantiles"].items()}, rel=1e-15)
    for k in ("episodes", "length_mean", "collision_rate", "boundary_rate", "timeout_rate", "remaining_mean", "dist_mean"):
        assert per[k] == whole[k], k


def test_summary_of_one_episode_and_of_none():
    from marbler_b200.policy import summarize_episodes
    s = summarize_episodes(_table([[(3.0, 7, 2, 0, 0, 1.0)]], 2))
    assert s["episodes"] == 1 and s["return_std"] == 0.0 and np.isnan(s["return_sem"])
    assert all(v == 3.0 for v in s["return_quantiles"].values())
    with pytest.raises(ValueError):
        summarize_episodes(_table([[], []], 2))


def _sharded_worker(rank, world, port, q):
    import torch.distributed as dist
    from marbler_b200.policy import summarize_episodes
    from marbler_b200.sharding import shard_range
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    rows = _sharded_rows()
    lo, n = shard_range(len(rows), rank, world)
    q.put((rank, summarize_episodes(_table(rows[lo:lo + n], 4), n_agents=2)))
    dist.destroy_process_group()


def _sharded_rows():
    rng = np.random.RandomState(3)
    return [[(float(rng.standard_normal() * 10), int(rng.randint(1, 82)), int(rng.randint(0, 4)), int(rng.randint(0, 2)),
              int(rng.randint(0, 7)), float(np.float32(rng.rand() * 5))) for _ in range(rng.randint(0, 5))]
            for _ in range(37)]


def test_sharded_summary_two_ranks_gloo_equals_one_rank():
    """Two gloo ranks with 19 and 18 envs of a hand-made table (envs with 0 .. K episodes) summarise the same episodes
    as one rank holding all 37 envs."""
    import torch.multiprocessing as mp
    from marbler_b200.policy import summarize_episodes
    want = summarize_episodes(_table(_sharded_rows(), 4), n_agents=2)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + ((os.getpid() + 1000) % 2000)
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted((q.get(timeout=120) for _ in procs), key=lambda x: x[0])
    [p.join(60) for p in procs]
    assert want["episodes"] > 37
    for rank, got in res:
        assert got == want, rank


# ------------------------------------------------------------------------------------------------ GPU

def _env(scenario, B, seed=11, env_id0=0, overrides=None):
    from marbler_b200 import config
    from marbler_b200.vec_env import VecEnv
    cfg = dict(config.load_yaml(config.default_config_path(scenario)), **(overrides or {}))
    return VecEnv(scenario, cfg, num_envs=B, device="cuda:0", seed=seed, env_id0=env_id0, auto_reset=True)


def _policy(env, scenario, overrides=None):
    from marbler_b200.policy import Policy
    sd = _checkpoint(CHECKPOINTS[scenario]) if scenario in CHECKPOINTS and not overrides else \
        _random_agent(env.N, env.D, env.n_actions)
    return Policy(sd, env.N, env.D, device="cuda:0")


def _explore(seed=9):
    from marbler_b200.policy import Exploration
    return Exploration("epsilon_greedy", seed=seed, eps_start=0.05, eps_finish=0.05, anneal_time=1, device="cuda:0")


def _rollout(scenario, B, K, use_graph=False, overrides=None, env_id0=0, record=None, seed=11):
    from marbler_b200.policy import EpisodeBatch, EvalLog, Rollout
    env = _env(scenario, B, seed=seed, env_id0=env_id0, overrides=overrides)
    batch = EpisodeBatch(env, record) if record else None
    return Rollout(env, _policy(env, scenario, overrides), use_graph=use_graph, steps_per_graph=4, explore=_explore(),
                   record=batch, evaluate=EvalLog(env, K))


class _Restated(object):
    """The accumulator rules of include/marbler_b200.h in float64 torch, fed from the env's buffers after each step."""

    def __init__(self, env, K):
        B, dev = env.B, env.device
        self.env, self.K = env, K
        self.table = {f: torch.zeros((B, K), dtype=torch.float64, device=dev) for f in FIELDS}
        self.count = torch.zeros((B,), dtype=torch.int64, device=dev)
        self.ret = torch.zeros((B,), dtype=torch.float64, device=dev)
        self.len = torch.zeros((B,), dtype=torch.int64, device=dev)
        self.dist = torch.zeros((B,), dtype=torch.float64, device=dev)

    def step(self):
        env = self.env
        team = torch.zeros((env.B,), dtype=torch.float32, device=env.device)
        d = torch.zeros((env.B,), dtype=torch.float64, device=env.device)
        for a in range(env.N):                       # agent index order, float32 and float64 adds one at a time
            team = team + env.reward[:, a]
            d = d + env.dist[:, a].double()
        self.ret += team.double()
        self.len += 1
        self.dist += d
        done = env.done != 0
        idx = (done & (self.count < self.K)).nonzero().squeeze(1)
        k = self.count[idx]
        msg = env.message[idx].long()
        for f, v in (("return", self.ret[idx]), ("length", self.len[idx].double()), ("message", msg.double()),
                     ("timeout", ((msg == 0) & (self.len[idx] > env.c.max_episode_steps)).double()),
                     ("remaining", env.remaining[idx].double()), ("dist", self.dist[idx].float().double())):
            self.table[f][idx, k] = v
        self.count[idx] += 1
        self.ret[done], self.len[done], self.dist[done] = 0.0, 0, 0.0


SCENARIOS = [("PredatorCapturePrey", None), ("PredatorCapturePrey", PCP20), ("Warehouse", None),
             ("MaterialTransport", None)]
IDS = ["PCP4", "PCP20", "Warehouse", "MaterialTransport"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario,overrides", SCENARIOS, ids=IDS)
def test_table_is_the_restatement_bit_for_bit(scenario, overrides):
    """1,024 envs, epsilon-greedy with eps = 0.05, K = 3, eager steps: after every env step the float64 torch
    restatement takes the same step; at the end of evaluate()'s K * (max_episode_steps + 1) steps every env has logged
    K episodes and every field equals the restatement (dist: the float32 rounding of the same float64 sum)."""
    K = 3
    ro = _rollout(scenario, 1024, K, overrides=overrides)
    env, log = ro.env, ro.eval_log
    ref = _Restated(env, K)
    log.begin()
    ro.reset()
    for _ in range(K * (env.c.max_episode_steps + 1)):
        ro.run(1)
        ref.step()
    torch.cuda.synchronize()
    assert bool((log.count == K).all())
    assert torch.equal(log.count.long(), ref.count)
    for f in FIELDS:
        assert torch.equal(log.data[f].double(), ref.table[f]), f
    assert log.return_.dtype == torch.float64 and torch.equal(log.return_, ref.table["return"])
    assert float(log.dist.sum()) > 0.0 and int(log.length.min()) >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("scenario,overrides", SCENARIOS, ids=IDS)
def test_table_agrees_with_the_env_statistics(scenario, overrides):
    """With K >= W steps no env can finish more episodes than it may log: the episodes that finished in the window
    are exactly the table's rows, and an episode still running at the end is in neither.  Counts and the length sum
    are equal; the return sum agrees to 1e-9 relative (the statistics add with atomics in arbitrary order).  The team
    kernels (7 or more robots) form the env's episode return with a warp butterfly instead of the in-order sum, so
    there each step's team reward may differ by the error bound of two float32 sums."""
    from marbler_b200 import _lib
    W = 120
    ro = _rollout(scenario, 1024, W, overrides=overrides)
    env, log = ro.env, ro.eval_log
    log.begin()
    ro.reset()
    env.stats.zero_()
    abs_sum = torch.zeros((), dtype=torch.float64, device="cuda:0")
    for _ in range(W):
        ro.run(1)
        abs_sum += env.reward.abs().double().sum()
    torch.cuda.synchronize()
    st = dict(zip(_lib.STAT_NAMES, env.stats.cpu().tolist()))
    valid = torch.arange(W, device="cuda:0")[None, :] < log.count[:, None].long()
    msg = log.message[valid].long()
    assert st["episodes"] == int(log.count.sum()) > 0
    assert st["collisions"] == int((msg & 1).ne(0).sum()) and st["boundary_exits"] == int((msg & 2).ne(0).sum())
    assert st["timeouts"] == int(log.timeout[valid].long().sum())
    assert st["length_sum"] == int(log.length[valid].long().sum())
    ret = float(log.return_[valid].sum())
    tol = 1e-9 * abs(ret)
    if env.N >= 7:
        tol += 2.0 * (env.N - 1) * 2.0 ** -24 * float(abs_sum)
    assert abs(st["return_sum"] - ret) <= tol, (st["return_sum"], ret)


def _same_run(a, b):
    for f in FIELDS + ("count",):
        assert torch.equal(a.eval_log.data[f], b.eval_log.data[f]), f
    for name in ("acc_return", "acc_length", "acc_dist"):
        assert torch.equal(getattr(a.eval_log, name), getattr(b.eval_log, name)), name
    assert torch.equal(a.env.state_f64, b.env.state_f64) and torch.equal(a.env.state_i32, b.env.state_i32)
    assert torch.equal(a.hidden, b.hidden) and torch.equal(a.env.obs, b.env.obs)


@pytest.mark.gpu
def test_graph_evaluate_equals_eager_with_and_without_recording():
    """PredatorCapturePrey, 1,024 envs, K = 2: evaluate() replayed from CUDA graphs equals eager launches bit for bit
    (table, counts, accumulators, env state, hidden state), with and without record= on the same Rollout; and a
    collect() records the same batch whether or not the rollout also evaluates."""
    from marbler_b200.policy import Rollout
    B, K, T = 1024, 2, 81
    for record in (None, T):
        g, e = (_rollout("PredatorCapturePrey", B, K, use_graph=u, record=record) for u in (True, False))
        for _ in range(2):
            g.evaluate(), e.evaluate()
        torch.cuda.synchronize()
        assert g._graph is not None
        assert bool((g.eval_log.count == K).all())
        _same_run(g, e)
    both = _rollout("PredatorCapturePrey", B, K, use_graph=True, record=T)
    plain = _rollout("PredatorCapturePrey", B, K, use_graph=True, record=T)
    only_record = Rollout(plain.env, plain.policy, use_graph=True, steps_per_graph=4, explore=plain.explore,
                          record=plain.record)
    got, want = both.collect(), only_record.collect()
    torch.cuda.synchronize()
    for f in want:
        assert torch.equal(got[f], want[f]), f
    assert torch.equal(both.env.state_f64, only_record.env.state_f64) and torch.equal(both.hidden, only_record.hidden)


@pytest.mark.gpu
def test_two_shards_log_what_one_batch_logs():
    B, K = 1024, 2
    halves = [_rollout("PredatorCapturePrey", B // 2, K, use_graph=True, env_id0=lo) for lo in (0, B // 2)]
    whole = _rollout("PredatorCapturePrey", B, K, use_graph=True)
    parts = [h.evaluate() for h in halves]
    w = whole.evaluate()
    torch.cuda.synchronize()
    for f in FIELDS + ("count",):
        assert torch.equal(w[f], torch.cat([p[f] for p in parts])), f


@pytest.mark.gpu
def test_first_episodes_are_the_recorded_episode_batch():
    """The shipped PCP vdn checkpoint, 4,096 envs, K = 1: return_mean is the mean of EpisodeBatch.reward.sum(1) of a
    collect() with episode_limit = max_episode_steps + 1 (no episode truncated), the same env seed and policy and a
    fresh Exploration of the same seed: the same episodes.  Not bit for bit (the float sums run in another order).
    The windowed env statistics over the same number of steps count every episode that finished in the window,
    short ones more often; their mean is printed, not asserted."""
    from marbler_b200.policy import EpisodeBatch, Rollout
    B = 4096
    ev = _rollout("PredatorCapturePrey", B, 1, use_graph=True)
    ev.evaluate()
    s = ev.eval_log.summary()
    T = ev.env.c.max_episode_steps + 1
    env = _env("PredatorCapturePrey", B)
    batch = EpisodeBatch(env, T)
    data = Rollout(env, _policy(env, "PredatorCapturePrey"), steps_per_graph=4, explore=_explore(), record=batch).collect()
    reward = data["reward"][:, :, 0].double().sum(1)
    assert bool((data["terminated"][:, :, 0].sum(1) == 1).all())
    assert s["episodes"] == B
    assert s["return_mean"] == pytest.approx(float(reward.mean()), rel=1e-6, abs=1e-9)
    lengths = data["filled"][:, 1:, 0].sum(1).double()
    assert s["length_mean"] == float(lengths.mean())
    win = _rollout("PredatorCapturePrey", B, 1, use_graph=True)
    win.reset()
    win.env.stats.zero_()
    win.run(T)
    st = win.env.read_stats()
    print("PCP vdn K=1 return_mean %.6f, windowed env.stats return_mean %.6f over %d episodes (%+.2f %%)" % (
        s["return_mean"], st["return_sum"] / st["episodes"], st["episodes"],
        100.0 * (st["return_sum"] / st["episodes"] / s["return_mean"] - 1.0)))


@pytest.mark.gpu
def test_eval_calls_check_their_arguments():
    """Every malformed table gives MRB_E_ARG, an unbound env MRB_E_STATE, without a launch and without touching the
    table; the well-formed calls are one launch each."""
    from marbler_b200 import _lib
    from marbler_b200.policy import EvalLog
    env = _env("PredatorCapturePrey", 64)
    lib, log = env.lib, EvalLog(env, 3)
    for t in log.data.values():
        t.fill_(5)
    for t in (log.acc_return, log.acc_length, log.acc_dist):
        t.fill_(5)
    snapshot = {k: v.clone() for k, v in list(log.data.items()) + [("acc", log.acc_return), ("accl", log.acc_length)]}

    def call(step, **kw):
        d = _lib.EvalTableDesc()
        C.memmove(C.byref(d), C.byref(log.desc), C.sizeof(d))
        for k, v in kw.items():
            setattr(d, k, v)
        return (lib.mrb_eval_step if step else lib.mrb_eval_begin)(env.handle, C.byref(d), None)

    cases = [(dict(struct_size=8), b"struct_size"), (dict(episodes=0), b"episodes"), (dict(episodes=-1), b"episodes"),
             (dict(episodes=(1 << 20) + 1), b"episodes")]
    cases += [(dict([(k, None)]), b"every pointer") for k, _ in _lib.EvalTableDesc._fields_[2:]]
    cases += [(dict([(k, getattr(log.desc, k) + off)]), b"aligned") for k, off in (
        ("return_", 4), ("acc_return", 4), ("acc_dist", 2), ("length", 2), ("remaining", 1), ("dist", 2),
        ("acc_length", 1), ("count", 3))]
    n0 = lib.mrb_launch_count()
    for step in (False, True):
        for kw, msg in cases:
            assert call(step, **kw) == MRB_E_ARG, (step, kw)
            assert msg in lib.mrb_last_error(env.handle), (step, kw, lib.mrb_last_error(env.handle))
        assert (lib.mrb_eval_step if step else lib.mrb_eval_begin)(env.handle, None, None) == MRB_E_ARG
    h = C.c_void_p()
    _lib.check(lib.mrb_create(C.byref(env.c), 0, 64, 0, C.byref(h)))
    assert lib.mrb_eval_begin(h, C.byref(log.desc), None) == MRB_E_STATE and b"mrb_bind" in lib.mrb_last_error(h)
    assert lib.mrb_eval_step(h, C.byref(log.desc), None) == MRB_E_STATE
    lib.mrb_destroy(h)
    assert lib.mrb_launch_count() == n0
    torch.cuda.synchronize()
    assert all(torch.equal(snapshot[k], v) for k, v in list(log.data.items()) + [("acc", log.acc_return),
                                                                              ("accl", log.acc_length)])
    # edge values of K are accepted: one launch each
    for K in (1, 1 << 20):
        d = _lib.EvalTableDesc()
        C.memmove(C.byref(d), C.byref(log.desc), C.sizeof(d))
        d.episodes = K
        assert lib.mrb_eval_begin(env.handle, C.byref(d), None) == 0
    log.begin()
    log.record()
    assert lib.mrb_launch_count() == n0 + 4
