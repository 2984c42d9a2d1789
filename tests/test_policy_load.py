"""Policy.load_state_dict / mrb_policy_load: new weights into an existing policy, in place, stream-ordered, capturable.

A policy holds its weights as device images in the layouts its kernels read (csrc/policy.cu policy_pack_kernel builds
them, at create and at load).  Loading W into a policy must leave it acting exactly as a policy created from W: every
word of every image rewritten (the policies loaded into here are created from all-NaN weights, so a word the load
missed shows up as NaN), in stream order with the acts around it, inside a captured graph, and under a captured
Rollout, whose graph keeps the policy's image pointers."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import golden_util as gu
import test_policy_kernels as tpk
from marbler_b200.policy import (check_state_dict, flatten_into, flatten_state_dict, state_dict_keys,
                                 state_dict_shapes)

SWEEP = [(k, s) for k, _, s in tpk.CASES]
MODELS = [("sweep-" + tpk._case_id((k, False, s)), s) for k, s in SWEEP] + [("fixture-" + n, None) for n in tpk.FIXTURES]


def _model(name, shape, seed=11):
    """(state_dict, shape) of a sweep case (random weights) or a checkpoint fixture."""
    if shape is None:
        _, sd, fs = tpk._fixture(name[len("fixture-"):])
        N = fs["N"]
        H, Din = sd[("agents.0." if fs["non_shared"] else "") + "fc1.weight"].shape
        A = sd[("agents.0." if fs["non_shared"] else "") + "fc2.weight"].shape[0]
        shape = dict(fs, H=H, A=A)
        assert Din == fs["D"] + (N if fs["agent_id"] else 0)
        return {k: np.asarray(v, dtype=np.float32) for k, v in sd.items()}, shape
    return tpk.random_model(shape, seed), shape


def _shapes_of(sd, N):
    _, f = flatten_state_dict(sd, N)
    return state_dict_shapes(N, f["non_shared"], f["use_rnn"], f["hidden_dim"], f["input_dim"], f["n_actions"])


def _perturbed(sd, seed, scale=0.05):
    rng = np.random.RandomState(seed)
    return {k: (v + scale * rng.standard_normal(v.shape)).astype(np.float32) for k, v in sd.items()}


# ------------------------------------------------------------------------------------------------ CPU

@pytest.mark.parametrize("shape", [tpk.S(128, True, 14, True, 3, 5, False), tpk.S(128, True, 14, True, 3, 5, True),
                                   tpk.S(64, False, 16, False, 3, 16, False), tpk.S(64, False, 16, False, 4, 24, True)],
                         ids=["gru-shared", "gru-per-agent", "linear-shared", "linear-per-agent"])
def test_device_flattening_equals_flatten_state_dict(shape):
    """flatten_into (what load_state_dict runs on the policy's device), run on CPU tensors of several dtypes and on
    numpy arrays, gives the bytes flatten_state_dict gives mrb_policy_create, in the same key order."""
    sd = tpk.random_model(shape, seed=3)
    flat, f = flatten_state_dict(sd, shape["N"])
    shapes = _shapes_of(sd, shape["N"])
    assert list(shapes) == state_dict_keys(shape["N"], shape["non_shared"], shape["use_rnn"])
    for conv in (lambda v: v, torch.from_numpy, lambda v: torch.from_numpy(v).double(),
                 lambda v: torch.from_numpy(v).requires_grad_()):
        out = torch.full((flat.size,), float("nan"))
        flatten_into({k: conv(v) for k, v in sd.items()}, shapes, out)
        assert np.array_equal(out.numpy().view(np.uint32), flat.view(np.uint32))
    half = {k: v.astype(np.float16) for k, v in sd.items()}
    out = torch.empty((flat.size,))
    flatten_into(half, shapes, out)
    assert np.array_equal(out.numpy(), flatten_state_dict(half, shape["N"])[0])


def test_validation_rejects_a_state_dict_of_another_shape():
    """Each mismatch raises ValueError naming the first key that differs, without touching a device."""
    N = 3
    gru = tpk.random_model(tpk.S(64, True, 10, True, N, 5, False), seed=1)
    shapes = _shapes_of(gru, N)
    check_state_dict(gru, shapes)
    check_state_dict({k: torch.from_numpy(v).half() for k, v in gru.items()}, shapes)

    def rejects(sd, key, shapes=shapes):
        with pytest.raises(ValueError, match=repr(key).replace(".", r"\.")):
            check_state_dict(sd, shapes)

    missing = dict(gru)
    del missing["rnn.bias_hh"]
    rejects(missing, "rnn.bias_hh")
    rejects(tpk.random_model(tpk.S(128, True, 10, True, N, 5, False), seed=1), "fc1.weight")          # hidden 128
    rejects(tpk.random_model(tpk.S(64, True, 10, True, N, 7, False), seed=1), "fc2.weight")           # 7 actions
    rejects(dict(gru, **{"fc2.bias": np.zeros(5, dtype=np.int64)}), "fc2.bias")                        # not a float
    rejects(dict(gru, extra=np.zeros(1, dtype=np.float32)), "extra")
    linear = tpk.random_model(tpk.S(64, False, 10, True, N, 5, False), seed=1)
    rejects(gru, "rnn.weight", shapes=_shapes_of(linear, N))                  # GRU weights for a Linear policy
    per_agent = tpk.random_model(tpk.S(64, True, 10, True, N, 5, True), seed=1)
    rejects(gru, "agents.0.fc1.weight", shapes=_shapes_of(per_agent, N))      # shared weights for a per-agent policy


# ------------------------------------------------------------------------------------------------ GPU helpers

DEV = torch.device("cuda:0")


def _act(pol, shape, B, seed=5):
    """One act from a random hidden state and observation, `fresh` on every 7th env: (q, h', actions)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    N, D, H, A = shape["N"], shape["D"], shape["H"], shape["A"]
    obs = torch.randn((B, N, D), generator=g, device=DEV)
    hid = torch.rand((B, N, H), generator=g, device=DEV) * 2 - 1
    fresh = (torch.arange(B, device=DEV) % 7 == 3).to(torch.uint8)
    q = torch.empty((B, N, A), device=DEV)
    a = pol.act(obs, hid, q=q, fresh=fresh)
    return q, hid, a


def _same(x, y):
    return all(torch.equal(u, v) for u, v in zip(x, y))


def _to_dev(sd):
    return {k: torch.as_tensor(v, device=DEV) for k, v in sd.items()}


# ------------------------------------------------------------------------------------------------ GPU: load == create

@pytest.mark.gpu
@pytest.mark.parametrize("accurate", [False, True], ids=["fp16", "accurate"])
@pytest.mark.parametrize("name,shape", MODELS, ids=[m[0] for m in MODELS])
def test_load_equals_create(name, shape, accurate):
    """A policy created from all-NaN weights, then loaded with W, acts bit for bit as a policy created from W; so does
    one loaded with W, W2, then W again."""
    sd, shape = _model(name, shape)
    kernel = tpk.expected_kernel(shape, accurate)
    nan = {k: np.full_like(v, np.nan) for k, v in sd.items()}
    loaded, created = tpk.make_policy(nan, shape, accurate), tpk.make_policy(sd, shape, accurate)
    loaded.load_state_dict(_to_dev(sd))
    w2 = _perturbed(sd, seed=1)
    for B in (1, 129, 4097):
        want = _act(created, shape, B)
        got = _act(loaded, shape, B)
        torch.cuda.synchronize()
        assert not torch.isnan(want[0]).any() and not torch.isnan(want[1]).any()
        assert _same(got, want), (name, kernel, B)
    loaded.load_state_dict(w2)
    other = _act(loaded, shape, 4097)
    torch.cuda.synchronize()
    assert not torch.equal(other[0], want[0])
    loaded.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})     # from the host this time
    assert _same(_act(loaded, shape, 4097), want)
    print("load == create: %s on %s" % (name, kernel))


@pytest.mark.gpu
def test_load_equals_create_on_the_mma_sync_kernel():
    """MRB_POLICY_TC=0 sends the tcgen05 shapes to the mma.sync kernel (tests/test_policy_kernels.py checks the
    routing), whose image the same load builds; the switch is read once per process, hence the subprocess."""
    env = dict(os.environ, MRB_POLICY_TC="0")
    res = subprocess.run([sys.executable, "-m", "pytest", __file__, "-q", "-s", "-m", "gpu", "-p", "no:cacheprovider",
                          "-k", "test_load_equals_create and tc2 and fp16 or test_load_equals_create and fixture and fp16"],
                         env=env, capture_output=True, text=True, timeout=900)
    print(res.stdout[-4000:])
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "passed" in res.stdout and " on mma" in res.stdout and " on tc2" not in res.stdout


# ------------------------------------------------------------------------------------------------ GPU: ordering, graphs

def _vdn():
    return _model("fixture-PredatorCapturePrey_vdn", None)


@pytest.mark.gpu
def test_load_is_stream_ordered_between_acts():
    """act with W0, load W1, act, all on one side stream with no synchronisation in between, at 65,536 envs: the first
    act sees W0 and the second W1."""
    sd0, shape = _vdn()
    sd1 = _perturbed(sd0, seed=2)
    w1 = _to_dev(sd1)
    B = 65536
    pol = tpk.make_policy(sd0, shape, False)
    want0, want1 = _act(tpk.make_policy(sd0, shape, False), shape, B), _act(tpk.make_policy(sd1, shape, False), shape, B)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got0 = _act(pol, shape, B)
        pol.load_state_dict(w1)
        got1 = _act(pol, shape, B)
    torch.cuda.synchronize()
    assert _same(got0, want0) and _same(got1, want1)
    assert not torch.equal(got0[0], got1[0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fixture-PredatorCapturePrey_vdn", "fixture-MaterialTransport_mappo_ns"])
def test_load_captured_in_a_graph_reads_the_tensors_at_replay(name):
    """load_state_dict from static device tensors (one of them float16) followed by act, captured in one CUDA graph
    (a synchronisation inside would break the capture); the static tensors changed in place between replays: each
    replay acts as a fresh policy of the tensors' values then.  Outside a graph, a load from device tensors makes
    torch synchronise nothing."""
    sd0, shape = _model(name, None)
    pol = tpk.make_policy(sd0, shape, False)
    B, N, D, H, A = 4097, shape["N"], shape["D"], shape["H"], shape["A"]
    static = _to_dev(sd0)
    half_key = list(static)[1]
    static[half_key] = static[half_key].half()
    g = torch.Generator(device=DEV).manual_seed(1)
    obs = torch.randn((B, N, D), generator=g, device=DEV)
    h0 = torch.rand((B, N, H), generator=g, device=DEV) - 0.5
    hid, q, act = h0.clone(), torch.empty((B, N, A), device=DEV), torch.empty((B, N), dtype=torch.int32, device=DEV)
    torch.cuda.set_sync_debug_mode("error")
    try:
        pol.load_state_dict(static)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                      # warm-up outside the capture
        pol.load_state_dict(static)
        pol.act(obs, hid, actions=act, q=q)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pol.load_state_dict(static)
        pol.act(obs, hid, actions=act, q=q)
    for seed in (7, 8):
        sd = _perturbed(sd0, seed=seed)
        for k, v in static.items():
            v.copy_(torch.as_tensor(sd[k]))
        sd[half_key] = sd[half_key].astype(np.float16)                  # what the half tensor holds
        hid.copy_(h0)
        graph.replay()
        ref = tpk.make_policy(sd, shape, False)
        rh, rq = h0.clone(), torch.empty((B, N, A), device=DEV)
        ra = ref.act(obs, rh, q=rq)
        torch.cuda.synchronize()
        assert torch.equal(q, rq) and torch.equal(hid, rh) and torch.equal(act, ra), seed


# ------------------------------------------------------------------------------------------------ GPU: captured rollouts

class TorchAgent(object):
    """RNNAgent / RNNNSAgent (utilities/rnn_agent.py, rnn_ns_agent.py) as plain torch parameters: the learner's copy."""

    def __init__(self, sd, N, D, agent_id):
        self.params = {k: torch.nn.Parameter(torch.as_tensor(v, device=DEV).clone()) for k, v in sd.items()}
        self.N, self.D, self.agent_id = N, D, agent_id
        self.ns = any(k.startswith("agents.") for k in sd)
        self.use_rnn = any(k.endswith("rnn.weight_ih") for k in sd)

    def state_dict(self):
        return dict(self.params)

    def forward(self, obs, h):
        """obs [B, N, D], h [B, N, H] -> q [B, N, A], h'"""
        qs, hs = [], []
        for i in range(self.N):
            w = lambda k: self.params[("agents.%d." % i if self.ns else "") + k]
            x = obs[:, i]
            if self.agent_id:
                x = torch.cat([x, torch.nn.functional.one_hot(torch.full((x.shape[0],), i, device=DEV), self.N).float()], 1)
            x = torch.relu(x @ w("fc1.weight").T + w("fc1.bias"))
            if self.use_rnn:
                hn = torch._VF.gru_cell(x, h[:, i], w("rnn.weight_ih"), w("rnn.weight_hh"), w("rnn.bias_ih"), w("rnn.bias_hh"))
            else:
                hn = torch.relu(x @ w("rnn.weight").T + w("rnn.bias"))
            qs.append(hn @ w("fc2.weight").T + w("fc2.bias"))
            hs.append(hn)
        return torch.stack(qs, 1), torch.stack(hs, 1)


def _learner_step(agent, data, D, steps=4):
    """One Adam step on a TD-like loss over the first `steps` rows of the recorded batch."""
    opt = torch.optim.Adam(list(agent.params.values()), lr=1e-2)
    obs, act, rew, filled = data["obs"], data["actions"], data["reward"], data["filled"]
    B, N, H = obs.shape[0], obs.shape[2], next(v for k, v in agent.params.items() if k.endswith("fc1.bias")).shape[0]
    h = torch.zeros((B, N, H), device=DEV)
    loss = 0
    for t in range(steps):
        q, h = agent.forward(obs[:, t, :, :D], h)
        chosen = q.gather(2, act[:, t]).squeeze(2).sum(1)
        loss = loss + (((chosen - rew[:, t, 0]) ** 2) * filled[:, t, 0]).mean()
    opt.zero_grad()
    loss.backward()
    opt.step()


ROLLOUTS = [  # (scenario, checkpoint, exploration mode, envs, episode limit)
    ("PredatorCapturePrey", "PredatorCapturePrey_vdn", "epsilon_greedy", 65536, 81),
    ("ArcticTransport", "ArcticTransport_qmix_ns", "epsilon_greedy", 2048, 40),
    ("MaterialTransport", "MaterialTransport_mappo_ns", "softmax", 2048, 40),
]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario,ckpt,mode,B,T", ROLLOUTS, ids=[r[1] for r in ROLLOUTS])
def test_captured_rollout_follows_the_learner(scenario, ckpt, mode, B, T):
    """collect() with W0; one optimiser step of a torch agent on the recorded batch; load_state_dict of the learner's
    parameters; collect() again on the same captured graph.  Both batches equal, bit for bit, those of fresh Policy and
    Rollout objects: one of W0 for the first, one of the learner's weights over an env and explorer brought to the
    same state for the second."""
    from marbler_b200 import config
    from marbler_b200.policy import EpisodeBatch, Exploration, Policy, Rollout
    from marbler_b200.vec_env import VecEnv
    sd0, shape = _model("fixture-" + ckpt, None)
    cfg = config.load_yaml(config.default_config_path(scenario))
    N, D = shape["N"], shape["D"]

    def env():
        return VecEnv(scenario, cfg, num_envs=B, device="cuda:0", seed=13, auto_reset=True)

    def explorer():
        return Exploration(mode, seed=4, eps_start=0.5, eps_finish=0.05, anneal_time=T, device="cuda:0")

    def rollout(vec, pol, ex):
        return Rollout(vec, pol, use_graph=True, steps_per_graph=8, explore=ex, record=EpisodeBatch(vec, T))

    ro = rollout(env(), Policy(sd0, N, D, device="cuda:0"), explorer())
    first = {k: v.clone() for k, v in ro.collect().items()}
    graph = ro._graph
    assert graph is not None
    agent = TorchAgent(sd0, N, D, shape["agent_id"])
    _learner_step(agent, first, D)
    new = agent.state_dict()
    assert all(v.is_cuda and v.requires_grad for v in new.values())
    assert not torch.equal(new["agents.0.fc2.bias" if agent.ns else "fc2.bias"].detach(),
                           torch.as_tensor(sd0["agents.0.fc2.bias" if agent.ns else "fc2.bias"], device=DEV))
    ro.policy.load_state_dict(new)
    second = ro.collect()
    assert ro._graph is graph
    torch.cuda.synchronize()

    vec, ex = env(), explorer()
    fresh0 = rollout(vec, Policy(sd0, N, D, device="cuda:0"), ex).collect()
    torch.cuda.synchronize()
    for k in first:
        assert torch.equal(first[k], fresh0[k]), ("first", k)
    w1 = {k: v.detach().cpu().numpy() for k, v in new.items()}
    fresh1 = rollout(vec, Policy(w1, N, D, device="cuda:0"), ex).collect()
    torch.cuda.synchronize()
    for k in second:
        assert torch.equal(second[k], fresh1[k]), ("second", k)
    assert not torch.equal(second["actions"], first["actions"])


# ------------------------------------------------------------------------------------------------ GPU: errors

@pytest.mark.gpu
def test_load_rejects_bad_arguments_and_leaves_the_policy_as_it_was():
    """Every mrb_policy_load argument error is MRB_E_ARG with a message, found before the device is touched; every
    load_state_dict shape error is a ValueError; after each the policy acts exactly as before."""
    from marbler_b200 import _lib
    from marbler_b200.policy import Rollout
    from marbler_b200.vec_env import VecEnv
    lib = _lib.load()
    sd, shape = _vdn()
    pol = tpk.make_policy(sd, shape, False)
    want = _act(pol, shape, 300)
    n = pol._staging.numel()
    good = torch.as_tensor(flatten_state_dict(_perturbed(sd, seed=3), shape["N"])[0], device=DEV)
    odd = torch.empty(n + 1, device=DEV)
    pinned = torch.empty(n, pin_memory=True)
    pinned.copy_(good.cpu())
    host = good.cpu().numpy()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cases = [(C.c_void_p(0), C.c_void_p(good.data_ptr()), n, "null policy"),
             (pol.handle, C.c_void_p(0), n, "null weights"),
             (pol.handle, C.c_void_p(good.data_ptr()), n - 1, "weights given"),
             (pol.handle, C.c_void_p(good.data_ptr()), n + 1, "weights given"),
             (pol.handle, C.c_void_p(odd.data_ptr() + 2), n, "4-byte aligned"),
             (pol.handle, C.c_void_p(pinned.data_ptr()), n, "device memory"),
             (pol.handle, host.ctypes.data_as(C.c_void_p), n, "device memory")]
    for handle, ptr, count, msg in cases:
        rc = lib.mrb_policy_load(handle, ptr, count, stream)
        assert rc == -1, msg
        err = lib.mrb_policy_last_error(handle if handle.value else None).decode()
        assert msg in err, (msg, err)
        torch.cuda.synchronize()
        assert _same(_act(pol, shape, 300), want), msg
    bad = [dict(sd, **{"fc1.bias": np.zeros(7, dtype=np.float32)}),
           {k: v for k, v in sd.items() if k != "rnn.bias_ih"},
           dict(sd, **{"fc2.weight": np.zeros((6, shape["H"]), dtype=np.float32)}),
           {"agents.%d.%s" % (i, k): v for i in range(shape["N"]) for k, v in sd.items()}]
    for b in bad:
        with pytest.raises(ValueError):
            pol.load_state_dict(_to_dev(b))
        torch.cuda.synchronize()
        assert _same(_act(pol, shape, 300), want)
    cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    ro = Rollout(VecEnv("PredatorCapturePrey", cfg, num_envs=64, device="cuda:0", seed=1), pol)
    with pytest.raises(AttributeError, match="load_state_dict"):
        ro.policy = tpk.make_policy(sd, shape, False)
    assert ro.policy is pol
