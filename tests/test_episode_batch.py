"""Episode recording into EPyMARL episode batches (mrb_record_begin / mrb_record_step, csrc/record.cu;
policy.EpisodeBatch, Rollout(record=).collect()).

Two restatements pin the contract of include/marbler_b200.h.  `RunnerBatch` is what EPyMARL's ParallelRunner.run
writes into its EpisodeBatch, one runner batch over a GymmaVecEnv; `ref_begin` / `ref_step` are the recorder's own
cursor rules, which start from any cursor state.  On the CPU a scripted fake env ties the two together; on the GPU
the kernel is compared with them element for element."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import golden_util as gu
from test_epymarl_adapter import _FakeWrapper

FIELDS = ("obs", "actions", "actions_onehot", "avail_actions", "reward", "terminated", "filled")
DTYPES = {"obs": np.float32, "actions": np.int64, "actions_onehot": np.float32, "avail_actions": np.int32,
          "reward": np.float32, "terminated": np.uint8, "filled": np.int64}
MRB_E_ARG, MRB_E_STATE = -1, -4
ENVS_PER_CTA = 32                     # record.cu kEnvs: the batch sweep straddles one tile


def shapes(B, T, N, W, A):
    R = T + 1
    return {"obs": (B, R, N, W), "actions": (B, R, N, 1), "actions_onehot": (B, R, N, A), "avail_actions": (B, R, N, A),
            "reward": (B, R, 1), "terminated": (B, R, 1), "filled": (B, R, 1)}


def team_reward(reward):
    """float32 sum of the agent rewards [B, N] in agent index order."""
    reward = np.asarray(reward, dtype=np.float32)
    s = reward[:, 0].copy()
    for a in range(1, reward.shape[1]):
        s = s + reward[:, a]
    return s


class RunnerBatch(object):
    """ParallelRunner.run's writes into its EpisodeBatch, restated (EPyMARL is not vendored): reset() stores the
    reset observation (zeros), avail_actions and filled in row 0; each step t stores, for the envs not terminated
    before it, the actions at t, reward and terminated (truncation included: the gym wrapper reports no episode_limit
    info) at t, and obs, avail_actions and filled at t + 1.  The terminal row's actions stay zero."""

    def __init__(self, B, T, N, W, A):
        self.T, self.A, self.t = T, A, 0
        self.b = {k: np.zeros(s, dtype=DTYPES[k]) for k, s in shapes(B, T, N, W, A).items()}
        self.b["avail_actions"][:, 0] = 1
        self.b["filled"][:, 0] = 1
        self.done = np.zeros(B, dtype=bool)

    def step(self, actions, obs, reward, terminated):
        """actions [B, N], obs [B, N, W] after the step, reward [B] (team), terminated [B] (done or time limit)."""
        b, t, live = self.b, self.t, ~self.done
        actions = np.asarray(actions)
        b["actions"][live, t, :, 0] = actions[live]
        b["actions_onehot"][live, t] = np.eye(self.A, dtype=np.float32)[actions[live]]
        b["reward"][live, t, 0] = np.asarray(reward, dtype=np.float32)[live]
        b["terminated"][live, t, 0] = np.asarray(terminated)[live]
        b["obs"][live, t + 1] = np.asarray(obs)[live]
        b["avail_actions"][live, t + 1] = 1
        b["filled"][live, t + 1] = 1
        self.done |= np.asarray(terminated, dtype=bool)
        self.t += 1


def ref_begin(b, cursor):
    T = b["obs"].shape[1] - 1
    b["obs"][:, 0] = 0
    b["avail_actions"][:, 0] = 1
    b["filled"][:, 0] = 1
    for k in ("actions", "actions_onehot", "reward", "terminated"):
        b[k][:, T] = 0
    cursor[:] = 0


def ref_step(b, cursor, obs, reward, done, actions):
    """One mrb_record_step on numpy arrays: cursor t (active) or ~t (terminated); t >= T writes nothing."""
    T, W, A = b["obs"].shape[1] - 1, b["obs"].shape[3], b["actions_onehot"].shape[3]
    D = obs.shape[2]
    active = cursor >= 0
    t = np.where(active, cursor, ~cursor)
    idx = np.nonzero(t < T)[0]
    te, act = t[idx], active[idx]
    a = np.where(act[:, None], actions[idx], 0)
    b["actions"][idx, te, :, 0] = a
    b["actions_onehot"][idx, te] = ((a[..., None] == np.arange(A)) & act[:, None, None]).astype(np.float32)
    b["reward"][idx, te, 0] = np.where(act, team_reward(reward[idx]), np.float32(0))
    term = act & ((done[idx] != 0) | (te + 1 >= T))
    b["terminated"][idx, te, 0] = term
    o = np.zeros((len(idx), obs.shape[1], W), dtype=np.float32)
    o[..., :D] = np.where(act[:, None, None], obs[idx], 0)
    b["obs"][idx, te + 1] = o
    b["avail_actions"][idx, te + 1] = act[:, None, None]
    b["filled"][idx, te + 1, 0] = act
    cursor[idx] = np.where(act & ~term, te + 1, ~(te + 1))


# ------------------------------------------------------------------------------------------------ CPU tests

def test_restated_runner_rules_on_a_scripted_env():
    """3 agents, declared width 6 over a 4-wide obs buffer, 5 actions; env 1 finishes on its own at step 1 (t = 2 of
    the fake), the others are cut by the time limit T = 3 at step 2."""
    from marbler_b200.epymarl import GymmaVecEnv
    B, T = 4, 3
    gym = GymmaVecEnv("robotarium_gym:Warehouse-v0", time_limit=T, num_envs=B, env=_FakeWrapper(B, done_at=1))
    gym.reset()
    N, W, A = gym.n_agents, gym.get_obs_size(), gym.get_total_actions()
    rb = RunnerBatch(B, T, N, W, A)
    b = {k: np.full(s, 7, dtype=DTYPES[k]) for k, s in shapes(B, T, N, W, A).items()}     # garbage: all overwritten
    cursor = np.full(B, 12345, dtype=np.int32)
    ref_begin(b, cursor)
    rng = np.random.RandomState(0)
    for t in range(T):
        actions = rng.randint(0, 3, size=(B, N))
        reward, term, _ = gym.step(torch.as_tensor(actions, dtype=torch.int32))
        per_agent = np.tile(np.array([1.0, 2.0, 3.5], dtype=np.float32), (B, 1))
        assert np.array_equal(team_reward(per_agent), reward.numpy())
        rb.step(actions, gym.get_obs().numpy(), team_reward(per_agent), term.numpy())
        done = ((np.arange(B) == 1) & (t == 1)).astype(np.uint8)         # the env's own done, without the limit
        ref_step(b, cursor, gym.get_obs().numpy()[..., :4], per_agent, done, actions)
    r = rb.b
    # row 0: the zero reset observation, every action available, filled
    assert not r["obs"][:, 0].any() and (r["avail_actions"][:, 0] == 1).all() and (r["filled"][:, 0] == 1).all()
    # env 1: terminal row 2 is filled and holds the terminal observation, but no action, reward or terminated
    assert r["terminated"][1, :, 0].tolist() == [0, 1, 0, 0] and r["filled"][1, :, 0].tolist() == [1, 1, 1, 0]
    assert not r["actions"][1, 2:].any() and not r["actions_onehot"][1, 2:].any() and r["reward"][1, 2:, 0].tolist() == [0, 0]
    assert (r["obs"][1, 2, :, :4] == 2.0).all() and not r["obs"][1, 3].any() and not r["avail_actions"][1, 3].any()
    # the others: truncation at the time limit is stored as terminal; rows 0 .. T are filled, row T has no action
    assert r["terminated"][[0, 2, 3], :, 0].tolist() == [[0, 0, 1, 0]] * 3 and (r["filled"][[0, 2, 3]] == 1).all()
    assert not r["actions"][:, T].any() and not r["reward"][:, T].any() and (r["obs"][[0, 2, 3], 3, :, :4] == 3.0).all()
    assert np.array_equal(r["actions_onehot"][0, 0].argmax(axis=1), r["actions"][0, 0, :, 0])
    assert r["reward"][0, :T, 0].tolist() == [6.5] * 3
    # zero tails: columns D .. W-1 of every row
    assert not r["obs"][..., 4:].any()
    # the recorder's cursor rules write the same batch over the garbage it started from
    for k in FIELDS:
        assert np.array_equal(b[k], r[k]), k
    assert cursor.tolist() == [~T] * B                  # inactive envs' cursors advance too


def test_record_calls_reject_null_arguments():
    from marbler_b200 import _lib, build
    build.build()
    lib = _lib.load()
    d = _lib.EpisodeBatchDesc(C.sizeof(_lib.EpisodeBatchDesc), 3, 16, 0, *([4096] * 9))
    assert lib.mrb_record_begin(None, C.byref(d), None) == MRB_E_ARG and b"env is NULL" in lib.mrb_last_error(None)
    assert lib.mrb_record_step(None, C.byref(d), C.c_void_p(4096), None) == MRB_E_ARG


# ------------------------------------------------------------------------------------------------ GPU: kernel alone

def _pcp_env(N, B, **kw):
    from marbler_b200 import config
    from marbler_b200.vec_env import VecEnv
    cfg = dict(config.load_yaml(config.default_config_path("PredatorCapturePrey")), predator=N // 2, capture=N - N // 2,
               num_neighbors=3)
    if N > 13:                                       # a spawn grid with room for the team and at most 64 cells
        cfg.update(ROBOT_INIT_RIGHT_THRESH=0.1, start_dist=0.25 if N > 20 else 0.3)
    return VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", **kw)


class _Canaried(object):
    """The batch tensors as views into buffers 64 elements longer, the tail set to a canary, and their desc."""

    def __init__(self, B, T, N, W, A, garbage=True, seed=0):
        from marbler_b200 import _lib
        g = torch.Generator(device="cuda:0").manual_seed(seed)
        self.shapes = shapes(B, T, N, W, A)
        self.buf, self.t = {}, {}
        for k, s in self.shapes.items():
            n = int(np.prod(s))
            tdt = getattr(torch, np.dtype(DTYPES[k]).name)
            raw = torch.randint(0, 100, (n + 64,), generator=g, device="cuda:0").to(tdt) if garbage else \
                torch.zeros((n + 64,), dtype=tdt, device="cuda:0")
            raw[n:] = 99
            self.buf[k], self.t[k] = raw, raw[:n].view(s)
        self.cursor_buf = torch.full((B + 64,), 99, dtype=torch.int32, device="cuda:0")
        self.cursor = self.cursor_buf[:B]
        self.desc = _lib.EpisodeBatchDesc(C.sizeof(_lib.EpisodeBatchDesc), T, W, 0, *[x.data_ptr() for x in (
            self.t["obs"], self.t["obs"], self.t["actions"], self.t["actions_onehot"], self.t["avail_actions"],
            self.t["reward"], self.t["terminated"], self.t["filled"], self.cursor)])

    def numpy(self):
        return {k: v.cpu().numpy() for k, v in self.t.items()}, self.cursor.cpu().numpy()

    def canaries_intact(self):
        n = {k: int(np.prod(s)) for k, s in self.shapes.items()}
        return all(bool((self.buf[k][n[k]:] == 99).all()) for k in self.buf) and bool((self.cursor_buf[-64:] == 99).all())


def _synthetic_step(env, rng, A):
    B, N, D = env.B, env.N, env.D
    obs = rng.standard_normal((B, N, D)).astype(np.float32)
    reward = (rng.standard_normal((B, N)) * 10).astype(np.float32)
    done = (rng.rand(B) < 0.2).astype(np.uint8)
    actions = rng.randint(0, A, size=(B, N)).astype(np.int32)
    env.obs.copy_(torch.as_tensor(obs))
    env.reward.copy_(torch.as_tensor(reward))
    env.done.copy_(torch.as_tensor(done))
    return obs, reward, done, torch.as_tensor(actions, device="cuda:0")


def _record(env, cb, actions=None):
    from marbler_b200 import _lib
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = env.lib.mrb_record_begin(env.handle, C.byref(cb.desc), s) if actions is None else \
        env.lib.mrb_record_step(env.handle, C.byref(cb.desc), C.c_void_p(actions.data_ptr()), s)
    _lib.check(rc, env.handle)


def _width(N, D):
    return D if N == 4 else D + (1 if N % 2 else 3)          # N*W*4 is not a multiple of 16 unless N == 4


def _one_step_case(N, B, T, seed):
    env = _pcp_env(N, B)
    A, D = env.n_actions, env.D
    W = _width(N, D)
    rng = np.random.RandomState(seed)
    cb = _Canaried(B, T, N, W, A, seed=seed)
    # cursors in every state: active at any row, terminated after any row, and past the end either way
    t = rng.randint(0, T + 1, size=B)
    cur = np.where(rng.rand(B) < 0.5, t, ~t).astype(np.int32)
    cur[rng.rand(B) < 0.1] = np.int32(2 ** 31 - 1)
    cur[rng.rand(B) < 0.05] = np.int32(-2 ** 31)
    cb.cursor.copy_(torch.as_tensor(cur))
    b, cursor = cb.numpy()
    obs, reward, done, actions = _synthetic_step(env, rng, A)
    _record(env, cb, actions)
    ref_step(b, cursor, obs, reward, done, actions.cpu().numpy())
    got, gcur = cb.numpy()
    for k in FIELDS:
        assert np.array_equal(got[k], b[k]), (k, N, B, T)
    assert np.array_equal(gcur, cursor) and cb.canaries_intact()


@pytest.mark.gpu
@pytest.mark.parametrize("N", [2, 3, 4, 5, 6, 8, 13, 20, 32])
def test_record_step_is_the_restatement_over_team_sizes(N):
    for T in (1, 2, 81):
        _one_step_case(N, ENVS_PER_CTA + 1, T, seed=N * 100 + T)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, ENVS_PER_CTA - 1, ENVS_PER_CTA, ENVS_PER_CTA + 1, 4097])
def test_record_step_is_the_restatement_over_batch_sizes(B):
    for N in (3, 4):
        for T in (1, 2, 81):
            _one_step_case(N, B, T, seed=B + N + T)


@pytest.mark.gpu
@pytest.mark.parametrize("N,B,T", [(3, 33, 81), (4, 4097, 2), (13, 257, 1), (20, 31, 5)])
def test_begin_and_t_steps_fill_the_runner_batch(N, B, T):
    """Begin over garbage, then T synthetic steps: the batch is the restated runner's, every row written once; later
    calls write nothing."""
    env = _pcp_env(N, B)
    A, D = env.n_actions, env.D
    W = _width(N, D)
    cb = _Canaried(B, T, N, W, A, seed=T)
    _record(env, cb)
    rb = RunnerBatch(B, T, N, W, A)
    rng = np.random.RandomState(N)
    for t in range(T):
        obs, reward, done, actions = _synthetic_step(env, rng, A)
        _record(env, cb, actions)
        term = (done != 0) | (t + 1 >= T)
        rb.step(actions.cpu().numpy(), np.pad(obs, ((0, 0), (0, 0), (0, W - D))), team_reward(reward), term)
    got, cursor = cb.numpy()
    for k in FIELDS:
        assert np.array_equal(got[k], rb.b[k]), k
    assert (cursor == ~T).all()                                  # inactive envs' cursors advance to the end too
    _synthetic_step(env, rng, A)
    _record(env, cb, actions)
    again, cursor2 = cb.numpy()
    assert all(np.array_equal(again[k], got[k]) for k in FIELDS) and np.array_equal(cursor2, cursor)
    assert cb.canaries_intact()


@pytest.mark.gpu
def test_record_calls_check_their_arguments():
    from marbler_b200 import _lib
    env = _pcp_env(4, 64)
    lib, A = env.lib, env.n_actions
    cb = _Canaried(64, 5, 4, env.D, A, garbage=False)
    act = torch.zeros((64, 4), dtype=torch.int32, device="cuda:0")
    snapshot = {k: v.clone() for k, v in cb.buf.items()}

    def call(step, **kw):
        d = _lib.EpisodeBatchDesc()
        C.memmove(C.byref(d), C.byref(cb.desc), C.sizeof(d))
        for k, v in kw.items():
            setattr(d, k, v)
        if step:
            return lib.mrb_record_step(env.handle, C.byref(d), C.c_void_p(act.data_ptr()), None)
        return lib.mrb_record_begin(env.handle, C.byref(d), None)

    cases = [(dict(struct_size=8), b"struct_size"), (dict(episode_limit=0), b"episode_limit"),
             (dict(episode_limit=-3), b"episode_limit"), (dict(obs_width=env.D - 1), b"obs_width"),
             (dict(obs_width=70000), b"obs_width"), (dict(state=cb.t["obs"].data_ptr() + 4), b"state must be obs")]
    cases += [(dict([(k, None)] + ([("state", None)] if k == "obs" else [])), b"every pointer") for k in (
        "obs", "state", "actions", "actions_onehot", "avail_actions", "reward", "terminated", "filled", "cursor")]
    cases += [(dict([(k, getattr(cb.desc, k) + off)] + ([("state", cb.desc.obs + off)] if k == "obs" else [])), b"aligned")
              for k, off in (("actions", 4), ("filled", 4), ("obs", 2), ("actions_onehot", 1), ("avail_actions", 2),
                             ("reward", 2), ("cursor", 1))]
    for step in (False, True):
        for kw, msg in cases:
            assert call(step, **kw) == MRB_E_ARG, (step, kw)
            assert msg in lib.mrb_last_error(env.handle), (step, kw, lib.mrb_last_error(env.handle))
    s = C.c_void_p(0)
    assert lib.mrb_record_begin(env.handle, None, s) == MRB_E_ARG
    assert lib.mrb_record_step(env.handle, C.byref(cb.desc), None, s) == MRB_E_ARG
    assert lib.mrb_record_step(env.handle, C.byref(cb.desc), C.c_void_p(act.data_ptr() + 2), s) == MRB_E_ARG
    # an env without bound buffers
    h = C.c_void_p()
    _lib.check(lib.mrb_create(C.byref(env.c), 0, 64, 0, C.byref(h)))
    assert lib.mrb_record_begin(h, C.byref(cb.desc), s) == MRB_E_STATE and b"mrb_bind" in lib.mrb_last_error(h)
    assert lib.mrb_record_step(h, C.byref(cb.desc), C.c_void_p(act.data_ptr()), s) == MRB_E_STATE
    lib.mrb_destroy(h)
    torch.cuda.synchronize()
    assert all(torch.equal(snapshot[k], cb.buf[k]) for k in snapshot)            # nothing reached the device


# ------------------------------------------------------------------------------------------------ GPU: closed loop

def _checkpoint(name):
    z = np.load(os.path.join(gu.GOLDEN, "policy", name + ".npz"))
    return {k[3:]: z[k] for k in z.files if k.startswith("sd.")}


def _random_agent(N, D, A, H=64, seed=0):
    """RNNAgent weights (shared, GRU, one-hot agent id) for the scenarios without a shipped checkpoint."""
    rng = np.random.RandomState(seed)
    w = lambda *s: (rng.standard_normal(s) * 0.3).astype(np.float32)
    return {"fc1.weight": w(H, D + N), "fc1.bias": w(H), "rnn.weight_ih": w(3 * H, H), "rnn.weight_hh": w(3 * H, H),
            "rnn.bias_ih": w(3 * H), "rnn.bias_hh": w(3 * H), "fc2.weight": w(A, H), "fc2.bias": w(A)}


CHECKPOINTS = {"PredatorCapturePrey": "PredatorCapturePrey_vdn", "ArcticTransport": "ArcticTransport_qmix_ns",
               "MaterialTransport": "MaterialTransport_mappo_ns"}
PCP20 = dict(predator=10, capture=10, ROBOT_INIT_RIGHT_THRESH=0.1, num_neighbors=3)


def _explorer(mode, seed=5):
    from marbler_b200.policy import Exploration
    if mode == "greedy":
        return None
    return Exploration(mode, seed=seed, eps_start=0.5, eps_finish=0.05, anneal_time=20, device="cuda:0")


def _restated_runner(gym, pol, explore, T):
    """ParallelRunner.run over a GymmaVecEnv: the same policy loop as Rollout (zero hidden state and observation at
    an episode start), the batch written by RunnerBatch.  Returns it and GymmaVecEnv's own team rewards."""
    B, N, D = gym.num_envs, gym.n_agents, gym._env.vec.D
    gym.reset()
    rb = RunnerBatch(B, T, N, gym.get_obs_size(), gym.get_total_actions())
    hidden = pol.init_hidden(B)
    obs = torch.zeros((B, N, D), device="cuda:0")
    fresh = torch.ones((B,), dtype=torch.uint8, device="cuda:0")
    sums = np.zeros((B, T + 1), dtype=np.float32)
    maxabs = np.zeros((B, T + 1), dtype=np.float32)
    for t in range(T):
        actions = pol.act(obs, hidden, fresh=fresh, explore=explore)
        reward, term, _ = gym.step(actions)
        per_agent = gym._env.vec.reward.cpu().numpy()
        sums[:, t], maxabs[:, t] = reward.cpu().numpy(), np.abs(per_agent).max(axis=1)
        rb.step(actions.cpu().numpy(), gym.get_obs().cpu().numpy(), team_reward(per_agent), term.cpu().numpy())
        obs = gym.get_obs()[..., :D].contiguous()
        fresh = term.to(torch.uint8)
    return rb.b, sums, maxabs


def _closed_loop_case(scenario, mode, B, T, overrides=None):
    from marbler_b200.epymarl import GymmaVecEnv
    from marbler_b200.policy import EpisodeBatch, Policy, Rollout
    key = "robotarium_gym:%s-v0" % scenario
    kw = dict(time_limit=T, num_envs=B, seed=17, device="cuda:0", config_overrides=overrides)
    g1, g2 = GymmaVecEnv(key, **kw), GymmaVecEnv(key, **kw)
    vec = g1._env.vec
    N, D, A = vec.N, vec.D, vec.n_actions
    sd = _checkpoint(CHECKPOINTS[scenario]) if scenario in CHECKPOINTS and not overrides else _random_agent(N, D, A)
    pol = Policy(sd, N, D, device="cuda:0")
    batch = EpisodeBatch(vec, T)
    assert batch.obs_width == g1.get_obs_size()
    got = Rollout(vec, pol, explore=_explorer(mode), record=batch).collect()
    want, sums, maxabs = _restated_runner(g2, pol, _explorer(mode), T)
    got = {k: v.cpu().numpy() for k, v in got.items()}
    B_, R, N_, W = got["obs"].shape
    assert np.array_equal(got["state"], got["obs"].reshape(B_, R, N_ * W))
    for k in FIELDS:
        assert np.array_equal(got[k], want[k]), (scenario, mode, k)
    # GymmaVecEnv's reward.sum(1) may add in another order.  Two float32 summations of N terms differ by at most
    # 2 (N - 1) 2^-24 sum |r_i| <= 2 (N - 1) 2^-24 N max |r_i| (seen: 1 ulp of the sum, 1.0 for 20 agents of -0.05, which
    # is more than an ulp or two of the largest term)
    live = want["filled"][:, 1:, 0] == 1
    diff = np.abs(got["reward"][:, :T, 0] - sums[:, :T]).astype(np.float64)
    tol = 2.0 * (N - 1) * 2.0 ** -24 * N * maxabs[:, :T].astype(np.float64)
    assert (diff[live] <= tol[live]).all(), (scenario, mode)
    ended = want["terminated"][:, :, 0].any(axis=1)
    assert ended.all()
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", ["PredatorCapturePrey", "Warehouse", "MaterialTransport", "ArcticTransport", "Simple"])
def test_collect_is_the_restated_runner_over_the_adapter(scenario):
    from marbler_b200 import config
    T = config.load_yaml(config.default_config_path(scenario))["max_episode_steps"] // 2
    for mode in ("greedy", "epsilon_greedy", "softmax"):
        _closed_loop_case(scenario, mode, 1024, T)


@pytest.mark.gpu
def test_collect_on_the_20_robot_team_kernel():
    _closed_loop_case("PredatorCapturePrey", "epsilon_greedy", 64, 12, overrides=PCP20)


# ------------------------------------------------------------------------------------------------ GPU: graph, shards

def _pcp_rollout(B, T, use_graph, env_id0=0, mode="epsilon_greedy"):
    from marbler_b200.policy import EpisodeBatch, Policy, Rollout
    from marbler_b200.vec_env import VecEnv
    cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=21, env_id0=env_id0, auto_reset=True)
    return Rollout(env, Policy(_checkpoint("PredatorCapturePrey_vdn"), 4, 16, device="cuda:0"), use_graph=use_graph,
                   steps_per_graph=4, explore=_explorer(mode, seed=3), record=EpisodeBatch(env, T))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["epsilon_greedy", "softmax"])
def test_graph_collect_equals_eager_and_shards_equal_one_batch(mode):
    B, T = 1024, 13
    r1, r2 = _pcp_rollout(B, T, True, mode=mode), _pcp_rollout(B, T, False, mode=mode)
    for k in range(2):
        d1, d2 = r1.collect(), r2.collect()
        torch.cuda.synchronize()
        for f in d1:
            assert torch.equal(d1[f], d2[f]), (k, f)
    assert r1._graph is not None
    assert torch.equal(r1.env.state_f64, r2.env.state_f64) and torch.equal(r1.env.state_i32, r2.env.state_i32)
    assert torch.equal(r1.hidden, r2.hidden) and torch.equal(r1.env.obs, r2.env.obs)
    assert int(r1.explore.step.item()) == int(r2.explore.step.item()) == 2 * T
    halves = [_pcp_rollout(B // 2, T, True, env_id0=lo, mode=mode) for lo in (0, B // 2)]
    parts = [h.collect() for h in halves]
    whole = _pcp_rollout(B, T, True, mode=mode).collect()
    torch.cuda.synchronize()
    for f in whole:
        assert torch.equal(whole[f], torch.cat([p[f] for p in parts])), f


@pytest.mark.gpu
def test_record_off_changes_nothing():
    """The same rollout with and without recording: identical env state, obs, actions and hidden state."""
    from marbler_b200.policy import Rollout
    rec = _pcp_rollout(1024, 13, True)
    ro = _pcp_rollout(1024, 13, True)
    bare = Rollout(ro.env, ro.policy, use_graph=True, steps_per_graph=4, explore=_explorer("epsilon_greedy", seed=3))
    rec.collect()
    bare.reset()
    bare.run(13)
    torch.cuda.synchronize()
    assert torch.equal(rec.env.state_f64, bare.env.state_f64) and torch.equal(rec.env.state_i32, bare.env.state_i32)
    assert torch.equal(rec.env.obs, bare.env.obs) and torch.equal(rec.env.stats, bare.env.stats)
    assert torch.equal(rec.actions, bare.actions) and torch.equal(rec.hidden, bare.hidden)


# ------------------------------------------------------------------------------------------------ GPU: production size

@pytest.mark.gpu
def test_production_collect_equals_a_hand_driven_torch_recorder():
    """65,536 PredatorCapturePrey envs, T = 81, the shipped vdn checkpoint, epsilon-greedy: the graph collect() equals
    an eager loop that records with plain torch indexing, bit for bit; every record call is one launch."""
    from marbler_b200 import _lib
    B, T = 65536, 81
    ro = _pcp_rollout(B, T, True)
    ro.steps_per_graph = 16
    lib = _lib.load()
    got = ro.collect()
    torch.cuda.synchronize()

    ref = _pcp_rollout(B, T, False)
    rec, ref.record = ref.record, None
    env, N, D, A = ref.env, 4, 16, 5
    b = {k: torch.zeros_like(v) for k, v in rec.data.items() if k != "state"}
    b["avail_actions"][:, 0] = 1
    b["filled"][:, 0] = 1
    active = torch.ones(B, dtype=torch.bool, device="cuda:0")
    ref.reset()
    for t in range(T):
        ref.run(1)
        idx = active.nonzero().squeeze(1)
        a = ref.actions[idx].long()
        b["actions"][idx, t, :, 0] = a
        b["actions_onehot"][idx, t] = torch.nn.functional.one_hot(a, A).float()
        r = env.reward[idx]
        s = r[:, 0].clone()
        for k in range(1, N):
            s = s + r[:, k]
        b["reward"][idx, t, 0] = s
        term = (env.done[idx] != 0) | (t + 1 >= T)
        b["terminated"][idx, t, 0] = term.to(torch.uint8)
        b["obs"][idx, t + 1, :, :D] = env.obs[idx]
        b["avail_actions"][idx, t + 1] = 1
        b["filled"][idx, t + 1] = 1
        active[idx[term]] = False
    torch.cuda.synchronize()
    for k in b:
        assert torch.equal(got[k], b[k]), k
    assert int(got["terminated"][:, :T - 1].sum()) > 0             # some envs finished before the limit
    n0 = lib.mrb_launch_count()
    for _ in range(3):
        ro.record.record(ro.actions)
    assert lib.mrb_launch_count() - n0 == 3
