"""On-device policies and rollouts (SURVEY.md section 8f-1).

The reference evaluates a trained EPyMARL agent on the host, one env, one step at a time
(utilities/misc.py:134-221 run_env): append the one-hot agent id when the model config says `obs_agent_id`
(misc.py:161-162), `q, hs = model(obs, hs)`, `actions = argmax(q)`, `env.step(actions)`; `hs` is re-zeroed at
the start of every episode (misc.py:156).  `Policy` holds the same network (utilities/rnn_agent.py RNNAgent,
utilities/rnn_ns_agent.py RNNNSAgent; weights in their state_dict layout) behind `mrb_policy_act`, a fused CUDA
kernel over all agents of all envs, and `Rollout` chains it with `mrb_step` on one stream - optionally captured
in a CUDA graph - so a whole evaluation runs without a host round trip per step.
PyTorch is used for device memory and streams only; there is no CPU path.
"""
import ctypes as C
import json

import numpy as np
import torch

from . import _lib
from .config import obs_space_dim


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _is_ns(state_dict):
    return any(k.startswith("agents.") for k in state_dict)


def _param_names(use_rnn):
    """The parameters of one RNNAgent in mrb_policy_create's order (state_dict order, include/marbler_b200.h)."""
    return ["fc1.weight", "fc1.bias"] + \
        (["rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh"] if use_rnn else ["rnn.weight", "rnn.bias"]) + \
        ["fc2.weight", "fc2.bias"]


def state_dict_keys(n_agents, non_shared, use_rnn):
    """Every key of an RNNAgent (or, non_shared, RNNNSAgent) state_dict, in the order of the flat weights."""
    prefixes = ["agents.%d." % i for i in range(n_agents)] if non_shared else [""]
    return [p + n for p in prefixes for n in _param_names(use_rnn)]


def flatten_state_dict(state_dict, n_agents):
    """state_dict of RNNAgent / RNNNSAgent -> (flat float32 array in mrb_policy_create's order, facts)."""
    sd = {k: np.asarray(v.detach().cpu().numpy() if hasattr(v, "detach") else v, dtype=np.float32)
          for k, v in state_dict.items()}
    ns = _is_ns(sd)
    use_rnn = ("agents.0." if ns else "") + "rnn.weight_ih" in sd
    keys = state_dict_keys(n_agents, ns, use_rnn)
    for k in keys:
        if k not in sd:
            raise KeyError("state_dict has no %r (n_agents = %d)" % (k, n_agents))
    flat = np.concatenate([sd[k].reshape(-1) for k in keys]).astype(np.float32)
    hidden, input_dim = sd[keys[0]].shape
    return flat, dict(non_shared=ns, use_rnn=use_rnn, hidden_dim=int(hidden), input_dim=int(input_dim),
                      n_actions=int(sd[keys[0].replace("fc1.weight", "fc2.weight")].shape[0]))


def state_dict_shapes(n_agents, non_shared, use_rnn, hidden_dim, input_dim, n_actions):
    """{key: shape} of the state_dict a policy of these facts was created from, in the order of the flat weights."""
    H, D, A = hidden_dim, input_dim, n_actions
    one = {"fc1.weight": (H, D), "fc1.bias": (H,), "rnn.weight_ih": (3 * H, H), "rnn.weight_hh": (3 * H, H),
           "rnn.bias_ih": (3 * H,), "rnn.bias_hh": (3 * H,), "rnn.weight": (H, H), "rnn.bias": (H,),
           "fc2.weight": (A, H), "fc2.bias": (A,)}
    return {k: one[k.split(".", 2)[-1] if non_shared else k] for k in state_dict_keys(n_agents, non_shared, use_rnn)}


def check_state_dict(state_dict, shapes):
    """Raise ValueError, naming the first mismatching key, unless `state_dict` holds exactly the keys of `shapes`
    (state_dict_shapes) with those shapes and a floating-point dtype.  Touches no device."""
    for k, shape in shapes.items():
        if k not in state_dict:
            raise ValueError("state_dict has no %r, which this policy needs" % k)
        v = state_dict[k]
        if tuple(v.shape) != shape:
            raise ValueError("state_dict[%r] has shape %s, this policy needs %s" % (k, tuple(v.shape), shape))
        floating = v.is_floating_point() if isinstance(v, torch.Tensor) else np.issubdtype(np.asarray(v).dtype, np.floating)
        if not floating:
            raise ValueError("state_dict[%r] is %s, not a floating-point type" % (k, v.dtype))
    for k in state_dict:
        if k not in shapes:
            raise ValueError("state_dict has %r, which this policy does not have" % k)


def flatten_into(state_dict, keys, out):
    """Copy the tensors (or numpy arrays) named by `keys`, flattened and converted to float32, back to back into the
    float32 vector `out` on its device, as flatten_state_dict orders them.  Tensors already on out's device are
    concatenated there without a synchronisation; the others are copied there first."""
    ts = [torch.as_tensor(state_dict[k]).detach().reshape(-1) for k in keys]
    ts = [t if t.device == out.device else t.to(out.device) for t in ts]
    torch.cat(ts, out=out)
    return out


class Policy(object):
    """Greedy (argmax-q) policy on the GPU.  obs_dim / n_agents describe the env's obs buffer [B, N, D]."""

    def __init__(self, state_dict, n_agents, obs_dim, obs_agent_id=None, device=None, accurate=False):
        """accurate=True: float32 arithmetic like the reference's own forward pass (csrc/policy_f32.cuh) - the greedy
        actions of a checkpoint are then the reference's, at ~10x the time of the FP16 tensor-core kernels."""
        if not torch.cuda.is_available():
            raise RuntimeError("marbler_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        flat, f = flatten_state_dict(state_dict, n_agents)
        if obs_agent_id is None:                         # misc.py:161: the model config decides; infer when not given
            obs_agent_id = f["input_dim"] == obs_dim + n_agents
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        self.n_agents, self.obs_dim, self.hidden_dim, self.n_actions = n_agents, obs_dim, f["hidden_dim"], f["n_actions"]
        self.obs_agent_id, self.use_rnn, self.non_shared = bool(obs_agent_id), f["use_rnn"], f["non_shared"]
        d = _lib.PolicyDesc(C.sizeof(_lib.PolicyDesc), obs_dim, f["input_dim"], f["hidden_dim"], f["n_actions"], n_agents,
                            int(self.obs_agent_id), int(self.use_rnn), int(self.non_shared), int(bool(accurate)))
        self.accurate = bool(accurate)
        self.handle = C.c_void_p()
        _lib.check_policy(self.lib.mrb_policy_create(C.byref(d), index, flat.ctypes.data_as(C.c_void_p), flat.size,
                                                     C.byref(self.handle)))
        self._shapes = state_dict_shapes(n_agents, self.non_shared, self.use_rnn, self.hidden_dim, f["input_dim"],
                                         self.n_actions)
        self._staging = torch.empty((flat.size,), dtype=torch.float32, device=self.device)

    @classmethod
    def from_files(cls, weights_path, model_config_path, n_agents, obs_dim, device=None, accurate=False):
        """The reference's own artefacts: a `.th` state_dict and the sacred model json next to it
        (scenarios/<S>/models/, loaded by utilities/misc.py:66-95 load_env_and_model)."""
        sd = torch.load(weights_path, map_location="cpu")
        with open(model_config_path) as fh:
            mc = json.load(fh)
        return cls(sd, n_agents, obs_dim, obs_agent_id=bool(mc.get("obs_agent_id", False)), device=device, accurate=accurate)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.mrb_policy_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def load_state_dict(self, state_dict):
        """Replace the weights in place: EPyMARL's mac.load_state(learner_mac) for the policy that collects.

        `state_dict` is an RNNAgent / RNNNSAgent state_dict of the shape this policy was created with (hidden size, input
        width, actions, GRU or Linear, shared or per-agent, n_agents; ValueError naming the first mismatching key
        otherwise, before any device work).  Its tensors may be on any device, or numpy arrays, of any float dtype.
        They are flattened into a float32 buffer the policy owns, on the current stream of its device, and
        mrb_policy_load rebuilds the weight images from it in one launch.  Stream-ordered: with the tensors on the
        policy's device nothing synchronises, and the call can be captured in a CUDA graph (replays read the tensors'
        values at replay time).  A captured `Rollout` of this policy sees the new weights at its next replay."""
        check_state_dict(state_dict, self._shapes)
        with torch.cuda.device(self.device):
            flatten_into(state_dict, self._shapes, self._staging)
            _lib.check_policy(self.lib.mrb_policy_load(
                self.handle, _ptr(self._staging), self._staging.numel(),
                C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), self.handle)

    def init_hidden(self, num_envs):
        """rnn_agent.py:17-19 init_hidden: zeros, one row per agent."""
        return torch.zeros((num_envs, self.n_agents, self.hidden_dim), dtype=torch.float32, device=self.device)

    def act(self, obs, hidden, actions=None, q=None, fresh=None, explore=None):
        """obs f32 [B,N,D], hidden f32 [B,N,H] (updated in place) -> actions i32 [B,N] (greedy).  `fresh` u8 [B]:
        envs that start an episode (zero hidden state and observation).  `explore`: an `Exploration` that then
        replaces the greedy actions (softmax reads q, allocated here when not given).  Stream-ordered, no
        synchronisation."""
        B = obs.shape[0]
        assert obs.is_cuda and obs.dtype == torch.float32 and obs.is_contiguous() and tuple(obs.shape) == (B, self.n_agents, self.obs_dim)
        assert hidden.dtype == torch.float32 and hidden.is_contiguous() and tuple(hidden.shape) == (B, self.n_agents, self.hidden_dim)
        if actions is None:
            actions = torch.empty((B, self.n_agents), dtype=torch.int32, device=self.device)
        if fresh is not None:
            assert fresh.dtype == torch.uint8 and fresh.is_contiguous() and fresh.shape == (B,)
        if explore is not None and explore.mode == "softmax" and q is None:
            q = torch.empty((B, self.n_agents, self.n_actions), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check_policy(self.lib.mrb_policy_act(
                self.handle, B, _ptr(obs), _ptr(hidden), _ptr(actions), _ptr(q), _ptr(fresh),
                C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), self.handle)
        if explore is not None:
            explore.select(actions, q, n_actions=self.n_actions)
        return actions


class Exploration(object):
    """EPyMARL's exploratory action selectors on the device (mrb_select_actions, csrc/explore.cu).

    mode "epsilon_greedy" is EpsilonGreedyActionSelector (QMIX, VDN, IQL) with its linear DecayThenFlatSchedule:
    eps(t) = max(eps_finish, eps_start - (eps_start - eps_finish) * t / anneal_time); each (env, agent) row keeps its
    greedy action or, with probability eps, takes one uniformly over all actions (MARBLER has no unavailable actions).
    mode "softmax" is SoftPoliciesSelector (MAPPO, IPPO): a draw from softmax(q).  The defaults are EPyMARL's.

    `step` is the schedule's counter t: an int64 CUDA tensor [1] that every `select` reads and then advances by one
    on the stream, so a captured CUDA graph moves it on at every replay.  EPyMARL's t_env counts env steps over the
    whole batch (it advances by the number of envs per step), so its `epsilon_anneal_time` is `anneal_time` times the
    batch size B here: anneal_time = epsilon_anneal_time / B.

    Every draw is a function of (seed, global env id, t, agent) alone (Philox; the exact contract is in
    include/marbler_b200.h): envs sharded over several devices draw what one device would have drawn when each
    shard passes the global id of its first env as `env_id0` (None: 0, or the env's own under `Rollout`)."""

    MODES = {"epsilon_greedy": _lib.SELECT_EPSILON_GREEDY, "softmax": _lib.SELECT_SOFTMAX}

    def __init__(self, mode, seed=0, env_id0=None, eps_start=1.0, eps_finish=0.05, anneal_time=50000, device=None):
        if mode not in self.MODES:
            raise ValueError("Exploration mode must be one of %s, not %r" % (sorted(self.MODES), mode))
        if not torch.cuda.is_available():
            raise RuntimeError("marbler_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.mode, self.seed, self.env_id0 = mode, int(seed) & (2 ** 64 - 1), env_id0
        self.eps_start, self.eps_finish, self.anneal_time = float(eps_start), float(eps_finish), int(anneal_time)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.step = torch.zeros((1,), dtype=torch.int64, device=self.device)

    def select(self, actions, q=None, n_actions=None):
        """actions i32 [B,N] on the device: the greedy actions on entry (epsilon_greedy, which needs `n_actions`)
        or output only (softmax, which reads q f32 [B,N,A]).  Advances `step` by one.  Stream-ordered."""
        B, N = actions.shape
        assert actions.dtype == torch.int32 and actions.is_contiguous() and actions.device == self.device
        if q is not None:
            assert q.dtype == torch.float32 and q.is_contiguous() and tuple(q.shape[:2]) == (B, N) and q.device == self.device
            n_actions = q.shape[2] if n_actions is None else n_actions
            assert q.shape[2] == n_actions
        if n_actions is None:
            raise ValueError("Exploration.select: pass n_actions (or q)")
        d = _lib.SelectDesc(C.sizeof(_lib.SelectDesc), self.MODES[self.mode], self.seed, int(self.env_id0 or 0),
                            self.eps_start, self.eps_finish, self.anneal_time)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrb_select_actions(
                self.device.index, B, N, int(n_actions), C.byref(d), _ptr(self.step), _ptr(q), _ptr(actions),
                C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return actions

    def epsilon(self):
        """eps(t) of the current counter, computed on the host (synchronises; for logging)."""
        t = int(self.step.item())
        return max(self.eps_finish, self.eps_start - (self.eps_start - self.eps_finish) * t / self.anneal_time)


class EpisodeBatch(object):
    """EPyMARL's EpisodeBatch for one runner batch of `vec_env`, filled on the device (mrb_record_begin /
    mrb_record_step, csrc/record.cu; the exact contract is in include/marbler_b200.h).

    Each env records one episode from row 0, as ParallelRunner.reset() and run() do: row 0 holds the zero reset
    observation.  Step t writes into row t the actions sent, the team reward (float32 sum over agents in index order)
    and terminated (the env's own done or the time limit: truncation counts as terminal, since the gym wrapper reports
    no episode_limit info), and into row t + 1 the observation after the step.  `filled` marks rows 0 .. terminal; every
    other element is zero, the actions of the terminal row included (ParallelRunner also selects an action there,
    which the learners' masks drop).  `obs_width` (default: the declared observation width, what
    `GymmaVecEnv.get_obs_size()` returns) pads each agent's observation with zeros.

    `data` is EPyMARL's scheme: obs [B,T+1,N,W] f32, state [B,T+1,N*W] (a view of obs), actions [B,T+1,N,1] i64,
    actions_onehot [B,T+1,N,A] f32, avail_actions [B,T+1,N,A] i32, reward / terminated / filled [B,T+1,1] as f32 /
    u8 / i64.  `cursor` [B] is the recorder's per-env position."""

    def __init__(self, vec_env, episode_limit, obs_width=None):
        self.env, self.lib = vec_env, _lib.load()
        B, N, A, dev = vec_env.B, vec_env.N, vec_env.n_actions, vec_env.device
        self.episode_limit = T = int(episode_limit)
        self.obs_width = W = obs_space_dim(vec_env.scenario, vec_env.cfg, vec_env.c) if obs_width is None else int(obs_width)
        self.obs = torch.zeros((B, T + 1, N, W), dtype=torch.float32, device=dev)
        self.actions = torch.zeros((B, T + 1, N, 1), dtype=torch.int64, device=dev)
        self.actions_onehot = torch.zeros((B, T + 1, N, A), dtype=torch.float32, device=dev)
        self.avail_actions = torch.zeros((B, T + 1, N, A), dtype=torch.int32, device=dev)
        self.reward = torch.zeros((B, T + 1, 1), dtype=torch.float32, device=dev)
        self.terminated = torch.zeros((B, T + 1, 1), dtype=torch.uint8, device=dev)
        self.filled = torch.zeros((B, T + 1, 1), dtype=torch.int64, device=dev)
        self.cursor = torch.zeros((B,), dtype=torch.int32, device=dev)
        self.desc = _lib.EpisodeBatchDesc(C.sizeof(_lib.EpisodeBatchDesc), T, W, 0, *[t.data_ptr() for t in (
            self.obs, self.obs, self.actions, self.actions_onehot, self.avail_actions, self.reward, self.terminated,
            self.filled, self.cursor)])

    @property
    def data(self):
        B, R, N, W = self.obs.shape
        return {"obs": self.obs, "state": self.obs.view(B, R, N * W), "actions": self.actions,
                "actions_onehot": self.actions_onehot, "avail_actions": self.avail_actions, "reward": self.reward,
                "terminated": self.terminated, "filled": self.filled}

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)

    def begin(self):
        """Row 0 of every env (and the zero row T of actions, reward and terminated); cursors to 0.  One launch."""
        with torch.cuda.device(self.env.device):
            _lib.check(self.lib.mrb_record_begin(self.env.handle, C.byref(self.desc), self._stream()), self.env.handle)

    def record(self, actions):
        """Record the step the env just took with `actions` (i32 [B,N] on the device).  One launch, stream-ordered;
        after `episode_limit` calls further ones write nothing."""
        assert actions.dtype == torch.int32 and actions.is_contiguous() and actions.device == self.env.device
        assert tuple(actions.shape) == (self.env.B, self.env.N)
        with torch.cuda.device(self.env.device):
            _lib.check(self.lib.mrb_record_step(self.env.handle, C.byref(self.desc), _ptr(actions), self._stream()),
                       self.env.handle)


EVAL_FIELDS = ("return", "length", "message", "timeout", "remaining", "dist")
QUANTILES = (5, 25, 50, 75, 95)


def _gather_rows(rows, device):
    """Concatenate every rank's rows (float64 [n_rank, F]) in rank order (torch.distributed, when a process group of
    more than one rank exists; the ranks may hold different numbers of rows)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return rows
    dev = device if dist.get_backend() == "nccl" else torch.device("cpu")
    world = dist.get_world_size()
    n = torch.tensor([rows.shape[0]], dtype=torch.int64, device=dev)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(s.item()) for s in sizes]
    top = max(sizes)
    padded = torch.zeros((top, rows.shape[1]), dtype=torch.float64, device=dev)
    padded[:rows.shape[0]] = rows.to(dev)
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded)
    return torch.cat([p[:s] for p, s in zip(parts, sizes)])


def summarize_episodes(data, n_agents=1, per_agent=False):
    """Per-episode statistics of an evaluation table (`EvalLog.data`: [B,K] fields and count [B]; row k of env b is
    an episode iff k < count[b]).  Host-side: synchronises with the table's device.  With a torch.distributed process
    group the rows of every rank are gathered first (all_gather, rank order), so a sharded evaluation summarises the
    same episodes as one device holding all envs.

    `per_agent`: returns divided by n_agents, the reading run_env gives shared-reward scenarios (its eval-only
    `shared_reward` config key, SURVEY.md Appendix B; the reference's misc.py is not vendored here, so this restates
    it).  return_std is the population standard deviation (np.std, what EPyMARL logs as test_return_std); return_sem
    uses the sample standard deviation (ddof = 1; NaN for one episode); the quantiles interpolate linearly
    (np.quantile's default)."""
    count = data["count"].to(torch.int64)
    K = data["return"].shape[1]
    valid = torch.arange(K, device=count.device)[None, :] < count[:, None]
    rows = torch.stack([data[f][valid].to(torch.float64) for f in EVAL_FIELDS], dim=1)
    rows = _gather_rows(rows, count.device).cpu().numpy()
    n = rows.shape[0]
    if n == 0:
        raise ValueError("the evaluation table holds no finished episode")
    ret = rows[:, 0] / (n_agents if per_agent else 1)
    msg = rows[:, 2].astype(np.int64)
    s = {"episodes": n, "return_mean": float(ret.mean()), "return_std": float(ret.std()),
         "return_sem": float(ret.std(ddof=1) / np.sqrt(n)) if n > 1 else float("nan"),
         "return_quantiles": {q: float(v) for q, v in zip(QUANTILES, np.quantile(ret, [q / 100 for q in QUANTILES]))},
         "length_mean": float(rows[:, 1].mean()),
         "collision_rate": float(((msg & 1) != 0).mean()), "boundary_rate": float(((msg & 2) != 0).mean()),
         "timeout_rate": float(rows[:, 3].mean()), "remaining_mean": float(rows[:, 4].mean()),
         "dist_mean": float(rows[:, 5].mean())}
    s.update(test_return_mean=s["return_mean"], test_return_std=s["return_std"], test_ep_length_mean=s["length_mean"])
    return s


class EvalLog(object):
    """Per-episode evaluation results of `vec_env`, filled on the device (mrb_eval_begin / mrb_eval_step,
    csrc/eval.cu; the exact contract is in include/marbler_b200.h): what run_env (utilities/misc.py:134-221) prints
    and logs for each of its episodes, for the first `episodes_per_env` (K) episodes of every env.

    After every env step each env adds the team reward (float32 sum over agents in index order, as the thread-per-env
    step kernels form the env's own episode return), one step and the distance its agents travelled to running accumulators; when the env finishes
    an episode and has logged fewer than K, the next row of its table gets the episode's return, length, terminal
    message (bit 0 collision, bit 1 boundary), timeout flag, `remaining` (prey left for PredatorCapturePrey, load left
    for MaterialTransport, 0 elsewhere) and distance (0 without track_dist).  Lengths count from `begin()`, which is
    meant to go with a reset of every env (as `Rollout.evaluate()` does).

    `data`: return [B,K] f64, length [B,K] i32, message / timeout [B,K] u8, remaining [B,K] i32, dist [B,K] f32 and
    count [B] i32; row k of env b is valid iff k < count[b]."""

    def __init__(self, vec_env, episodes_per_env):
        self.env, self.lib = vec_env, _lib.load()
        B, dev = vec_env.B, vec_env.device
        self.episodes = K = int(episodes_per_env)
        self.return_ = torch.zeros((B, K), dtype=torch.float64, device=dev)
        self.length = torch.zeros((B, K), dtype=torch.int32, device=dev)
        self.message = torch.zeros((B, K), dtype=torch.uint8, device=dev)
        self.timeout = torch.zeros((B, K), dtype=torch.uint8, device=dev)
        self.remaining = torch.zeros((B, K), dtype=torch.int32, device=dev)
        self.dist = torch.zeros((B, K), dtype=torch.float32, device=dev)
        self.acc_return = torch.zeros((B,), dtype=torch.float64, device=dev)
        self.acc_length = torch.zeros((B,), dtype=torch.int32, device=dev)
        self.acc_dist = torch.zeros((B,), dtype=torch.float64, device=dev)
        self.count = torch.zeros((B,), dtype=torch.int32, device=dev)
        self.desc = _lib.EvalTableDesc(C.sizeof(_lib.EvalTableDesc), K, *[t.data_ptr() for t in (
            self.return_, self.length, self.message, self.timeout, self.remaining, self.dist, self.acc_return,
            self.acc_length, self.acc_dist, self.count)])

    @property
    def data(self):
        return {"return": self.return_, "length": self.length, "message": self.message, "timeout": self.timeout,
                "remaining": self.remaining, "dist": self.dist, "count": self.count}

    def _call(self, fn):
        with torch.cuda.device(self.env.device):
            _lib.check(fn(self.env.handle, C.byref(self.desc),
                          C.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)), self.env.handle)

    def begin(self):
        """Accumulators and counts to 0 (the rows stay as they are).  One launch, stream-ordered."""
        self._call(self.lib.mrb_eval_begin)

    def record(self):
        """Log the step the env just took.  One launch, stream-ordered, capturable."""
        self._call(self.lib.mrb_eval_step)

    def summary(self, per_agent=False):
        """summarize_episodes over this table (synchronises; gathers the ranks of a process group)."""
        return summarize_episodes(self.data, self.env.N, per_agent)


class Rollout(object):
    """run_env's loop for a whole batch, on the device: act -> step -> act -> ...  (misc.py:155-187).

    The env auto-resets finished envs inside the step kernel; their `done` flag doubles as the next step's
    `fresh` mask (zero hidden state, zero observation - what run_env feeds after env.reset()).

    `explore`: an `Exploration` that selects the actions of every step after the policy (its counter advances inside
    the captured graph too, and `reset` does not rewind it: the schedule runs across episodes).  When its `env_id0` is
    None it takes the env's own, so that the ranks of a sharded run draw distinct streams.

    `record`: an `EpisodeBatch` of the same env that records every step after it is taken (one more launch per step,
    captured in the graph too); `collect()` then fills it with one runner batch.

    `evaluate`: an `EvalLog` of the same env that logs every step after it is taken (one more launch per step, after
    the record launch, captured in the graph too); `evaluate()` then fills it with K episodes per env.

    `skip_finished`: step only the envs that `record` or `evaluate` still needs (mrb_step_masked), as EPyMARL's
    ParallelRunner steps only envs_not_terminated: with `record`, the envs whose recorded episode has not terminated
    (cursor >= 0); with `evaluate`, the envs that have logged fewer than K episodes; with both, either.  The mask is
    computed on the device before every step, inside the captured graph.  A `collect()` or `evaluate()` that starts
    from the same env state fills `record.data` / `evaluate.data` bit for bit as without it, with the same exploration
    draws; what differs is `env.stats` (it counts only the steps taken) and the state the skipped envs are left in: they
    stop where their last needed step left them instead of running on into episodes nobody reads, so their episode
    counters, which key the reset streams, do not advance, and the next call's `reset()` starts them in other episodes.
    Off by default; needs `record` or `evaluate`."""

    def __init__(self, vec_env, policy, use_graph=True, steps_per_graph=8, explore=None, record=None, evaluate=None,
                 skip_finished=False):
        if skip_finished and record is None and evaluate is None:
            raise ValueError("Rollout(skip_finished=True) needs record= or evaluate=: they decide which envs are finished")
        assert vec_env.N == policy.n_agents and vec_env.D == policy.obs_dim and vec_env.device == policy.device
        assert vec_env.n_actions == policy.n_actions, "policy and scenario disagree on the number of actions"
        self.env, self._policy = vec_env, policy
        self.hidden = policy.init_hidden(vec_env.B)
        self.actions = torch.zeros((vec_env.B, vec_env.N), dtype=torch.int32, device=vec_env.device)
        self.explore, self.q = explore, None
        if explore is not None:
            assert explore.device == vec_env.device
            if explore.env_id0 is None:
                explore.env_id0 = vec_env.env_id0
            if explore.mode == "softmax":
                self.q = torch.zeros((vec_env.B, vec_env.N, policy.n_actions), dtype=torch.float32, device=vec_env.device)
        assert record is None or record.env is vec_env, "the EpisodeBatch must belong to the rollout's env"
        self.record = record
        assert evaluate is None or evaluate.env is vec_env, "the EvalLog must belong to the rollout's env"
        self.eval_log = evaluate
        self.skip_finished = bool(skip_finished)
        # u8 [B] mask of the envs the next step takes, written through a bool view; with both record and evaluate the
        # second buffer holds evaluate's part
        self.active = torch.ones((vec_env.B,), dtype=torch.uint8, device=vec_env.device) if skip_finished else None
        self._eval_needs = torch.ones((vec_env.B,), dtype=torch.bool, device=vec_env.device) \
            if skip_finished and record is not None and evaluate is not None else None
        self.use_graph, self.steps_per_graph = use_graph, int(steps_per_graph)
        self._graph = None

    @property
    def policy(self):
        """The policy the rollout acts with.  A captured graph holds its weight images, so the policy cannot be
        replaced; `rollout.policy.load_state_dict(sd)` changes its weights in place, graph included."""
        return self._policy

    @policy.setter
    def policy(self, _):
        raise AttributeError("Rollout.policy cannot be replaced (a captured graph keeps acting with the old policy's "
                             "weights); load new weights with rollout.policy.load_state_dict(state_dict)")

    def reset(self):
        self.env.reset()
        self.env.done.fill_(1)          # every env starts an episode: first act() sees fresh = 1 everywhere
        self.hidden.zero_()

    def _update_active(self):
        """self.active = the envs `record` or `evaluate` still needs, from their cursors and counts (on the stream)."""
        a = self.active.view(torch.bool)
        if self.record is not None:
            torch.ge(self.record.cursor, 0, out=a)
            if self.eval_log is not None:
                torch.lt(self.eval_log.count, self.eval_log.episodes, out=self._eval_needs)
                a.logical_or_(self._eval_needs)
        else:
            torch.lt(self.eval_log.count, self.eval_log.episodes, out=a)
        return self.active

    def _one(self):
        self.policy.act(self.env.obs, self.hidden, actions=self.actions, q=self.q, fresh=self.env.done, explore=self.explore)
        self.env.step(self.actions, active=self._update_active() if self.skip_finished else None)
        if self.record is not None:
            self.record.record(self.actions)
        if self.eval_log is not None:
            self.eval_log.record()

    def collect(self):
        """One EPyMARL runner batch into `record`: mrb_record_begin, `reset()`, then exactly episode_limit env steps,
        so every env records one episode and the result is the same with or without the graph (the auto-resets of
        envs that finish early included).  No host synchronisation.  Returns `record.data`."""
        if self.record is None:
            raise ValueError("Rollout.collect needs record=EpisodeBatch(...)")
        self.record.begin()
        self.reset()
        self.run(self.record.episode_limit)
        return self.record.data

    def evaluate(self):
        """K episodes of every env into `evaluate` (its `episodes`): mrb_eval_begin, `reset()`, then
        K * (max_episode_steps + 1) env steps.  An episode ends after at most max_episode_steps + 1 steps, so at the end
        every env has logged exactly K episodes, whatever its episode lengths and with no host synchronisation on the
        way; the result does not depend on the graph, the batch size or the sharding.  Envs that have logged K episodes
        keep stepping until the end (unlogged), unless `skip_finished`.  Returns `evaluate.data`; `evaluate.summary()`
        reduces it."""
        if self.eval_log is None:
            raise ValueError("Rollout.evaluate needs evaluate=EvalLog(...)")
        self.eval_log.begin()
        self.reset()
        self.run(self.eval_log.episodes * (self.env.c.max_episode_steps + 1))
        return self.eval_log.data

    def run(self, steps):
        """Advance every env by `steps` env steps (2 kernels per step, 4 with `explore`, one more each with `record`
        and `evaluate`, one more and the mask's torch kernels with `skip_finished`; no host synchronisation)."""
        k = self.steps_per_graph
        if self.use_graph:
            if self._graph is None and steps > k:
                self._one()                                   # warm-up outside capture
                steps -= 1
                torch.cuda.synchronize(self.env.device)
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):           # capture records k steps; it does not run them
                    for _ in range(k):
                        self._one()
            while self._graph is not None and steps >= k:
                self._graph.replay()
                steps -= k
        for _ in range(steps):
            self._one()
