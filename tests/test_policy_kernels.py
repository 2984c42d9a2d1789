"""The three policy kernels against a float64 restatement of RNNAgent.forward, over the shapes mrb_policy_create
accepts, at production batch sizes, and at the edges where such kernels go wrong.

Which kernel serves a model (mrb_policy_act, csrc/policy.cu):
  * Policy(..., accurate=True)                       -> float32 kernel (csrc/policy_f32.cuh), 16 envs per CTA;
  * hidden 128 + GRUCell with <= 8 actions          -> persistent tcgen05 / TMEM kernel (csrc/policy_tc2.cuh),
                                                       one CTA per SM looping over (128-env tile, agent) work items;
  * everything else, and every model under MRB_POLICY_TC=0 -> mma.sync kernel (policy_act_kernel), 64 envs per CTA.
Every case names the kernel it is meant to reach and `expected_kernel` restates the rule; in the shape sweep a
profiler trace of one launch shows the kernel that actually ran.

The reference `forward64` is float64 throughout.  With fp16=True it rounds to FP16 exactly what the tensor-core
kernels feed their MMAs (input incl. one-hot id, W1, relu(fc1), h, W_ih / W_hh, h' and W2); biases, the old h of the
GRU blend and all sums stay unrounded.  With fp16=False it is the plain network, the float32 kernel's contract.  It
is anchored without a GPU on the shipped-checkpoint fixtures (tests/golden/policy), whose float32 outputs come from
the reference's own agent classes.

Error bars are relative to the largest |q| of the reference (`scale`) and sit about 4x above the worst value measured
on a B200 (noted beside them), except where that would be looser than tests/test_policy.py's bars.  The median bar
catches contract errors that a max bar hides, such as an operand left unrounded (~1e-5 against FP32 noise of ~3e-8)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import golden_util as gu
from trace_util import kernels_launched

POLICY = os.path.join(gu.GOLDEN, "policy")
FIXTURES = ["ArcticTransport_qmix_ns", "MaterialTransport_mappo_ns", "PredatorCapturePrey_vdn"]

# per kernel: max |q - fc2_64(h')| < rel * |q_ref|max + floor, median |q - q_ref| / |q_ref|max, and
# max |h - h_ref| / max(1, |h_ref|max); measured on a B200 (1,000 W) beside each bar.  The h bar of the FP16 kernels is set
# by FP16 roundings that fall the other way in float64 (half an FP16 ulp of an operand): up to 4.7e-4 on the random models,
# 4.0e-3 on the shipped PredatorCapturePrey checkpoint over 262,144 agents, whose weights are larger.
Q_MAX = {"tc2": (2e-6, 0.0), "mma": (2e-6, 0.0), "f32": (2e-6, 0.0)}   # measured 3.2e-7 / 4.9e-7 / 5.0e-7
Q_MED = {"tc2": 2.5e-7, "mma": 2.5e-7, "f32": 3e-7}                   # measured 2.9e-8 / 6.5e-8 / 8.2e-8
H_MAX = {"tc2": 1.6e-2, "mma": 1.5e-3, "f32": 3e-6}                   # measured 4.0e-3 / 3.1e-4 / 6.8e-7
KERNEL_NAME = {"tc2": "policy_act_tc2_kernel", "mma": "policy_act_kernel<", "f32": "policy_act_f32_kernel"}


def forward64(sd, prefix, use_rnn, x, h, fp16):
    """utilities/rnn_agent.py:21-29 RNNAgent.forward in float64 on x's device: x [R, input_dim] (obs + one-hot id),
    h [R, H] -> (q [R, A], h' [R, H])."""
    dev = x.device
    r = (lambda t: t.half().double()) if fp16 else (lambda t: t.double())
    w = lambda k: r(torch.as_tensor(sd[prefix + k], device=dev))
    b = lambda k: torch.as_tensor(sd[prefix + k], device=dev).double()
    x, h = x.double(), h.double()
    x = torch.relu(r(x) @ w("fc1.weight").T + b("fc1.bias"))
    if use_rnn:
        H = h.shape[1]
        gi = r(x) @ w("rnn.weight_ih").T + b("rnn.bias_ih")
        gh = r(h) @ w("rnn.weight_hh").T + b("rnn.bias_hh")
        rg = torch.sigmoid(gi[:, :H] + gh[:, :H])
        zg = torch.sigmoid(gi[:, H:2 * H] + gh[:, H:2 * H])
        n = torch.tanh(gi[:, 2 * H:] + rg * gh[:, 2 * H:])
        hn = (1 - zg) * n + zg * h
    else:
        hn = torch.relu(r(x) @ w("rnn.weight").T + b("rnn.bias"))
    return r(hn) @ w("fc2.weight").T + b("fc2.bias"), hn


def step64(sd, shape, obs, h, fresh, fp16):
    """One env step of every agent: obs [B, N, D], h [B, N, H] (float64), fresh bool [B] or None -> q, h'."""
    N, D, agent_id, non_shared, use_rnn = shape["N"], shape["D"], shape["agent_id"], shape["non_shared"], shape["use_rnn"]
    obs, h = obs.double().clone(), h.double().clone()
    if fresh is not None:
        obs[fresh] = 0
        h[fresh] = 0
    qs, hs = [], []
    for i in range(N):
        x = obs[:, i]
        if agent_id:                                           # utilities/misc.py:161-162
            onehot = torch.zeros((x.shape[0], N), dtype=x.dtype, device=x.device)
            onehot[:, i] = 1
            x = torch.cat([x, onehot], dim=1)
        q, hn = forward64(sd, "agents.%d." % i if non_shared else "", use_rnn, x, h[:, i], fp16)
        qs.append(q), hs.append(hn)
    return torch.stack(qs, 1), torch.stack(hs, 1)


def fc2_64(sd, shape, h, fp16):
    """fc2 alone (rnn_agent.py:28) in float64 on h' [B, N, H]: q of the kernel's own h'."""
    r = (lambda t: t.half().double()) if fp16 else (lambda t: t.double())
    qs = []
    for i in range(shape["N"]):
        p = "agents.%d." % i if shape["non_shared"] else ""
        w = r(torch.as_tensor(sd[p + "fc2.weight"], device=h.device))
        qs.append(r(h[:, i].double()) @ w.T + torch.as_tensor(sd[p + "fc2.bias"], device=h.device).double())
    return torch.stack(qs, 1)


# ------------------------------------------------------------------------------------------------ the anchor (CPU)

def _fixture(name):
    z = np.load(os.path.join(POLICY, name + ".npz"))
    sd = {k[3:]: z[k] for k in z.files if k.startswith("sd.")}
    N, D = int(z["n_agents"]), int(z["obs_dim"])
    ns = any(k.startswith("agents.") for k in sd)
    pre = "agents.0." if ns else ""
    shape = dict(N=N, D=D, agent_id=bool(z["obs_agent_id"]), non_shared=ns, use_rnn=(pre + "rnn.weight_ih") in sd)
    return z, sd, shape


@pytest.mark.parametrize("name", FIXTURES)
def test_float64_reference_reproduces_the_fixtures(name):
    """forward64 against the float32 outputs of the reference's own classes: the plain network (`q`, `h`) and the
    network with FP16-rounded MMA operands (`q_tf32`, `h_tf32`), 4 recurrent steps.  The median difference is float32
    rounding of the fixtures (<= 2.7e-8 |q|max); a gate swap, a missing FP16 rounding or a misplaced one-hot id moves
    it to 7e-6 or more.  With FP16 rounding the worst element is larger: where a float32 and a float64 value fall on
    opposite sides of an FP16 rounding boundary the operands differ by half an FP16 ulp, and the recurrence carries that
    on."""
    z, sd, shape = _fixture(name)
    T, B = z["obs"].shape[:2]
    H = z["h"].shape[-1]
    # (max |q - q_fix|, median, max |h - h_fix|) bars, measured on the three fixtures beside them
    bars = {False: (1e-6, 1e-7, 8e-6),                         # measured 1.8e-7, 2.7e-8, 2.0e-6
            True: (1.5e-4, 1e-7, 1.5e-3)}                      # measured 3.7e-5, 2.1e-8, 3.5e-4
    for fp16, qk, hk in ((False, "q", "h"), (True, "q_tf32", "h_tf32")):
        h = torch.zeros((B, shape["N"], H), dtype=torch.float64)
        scale = float(np.abs(z[qk]).max())
        d = []
        for t in range(T):
            q, h = step64(sd, shape, torch.as_tensor(z["obs"][t]), h, None, fp16)
            d.append(np.abs(q.numpy() - z[qk][t]).ravel() / scale)
        d = np.concatenate(d)
        hs = max(1.0, float(np.abs(z[hk]).max()))
        herr = float(np.abs(h.numpy() - z[hk]).max()) / hs
        print("anchor %s fp16=%d: |q - %s| max %.2e median %.2e (|q|max), max |h - %s| = %.2e"
              % (name, fp16, qk, d.max(), np.median(d), hk, herr))
        qmax, qmed, hmax = bars[fp16]
        assert d.max() < qmax and np.median(d) < qmed and herr < hmax, (fp16, d.max(), np.median(d), herr)


# ------------------------------------------------------------------------------------------------ shared helpers

def expected_kernel(shape, accurate):
    """mrb_policy_act's routing (csrc/policy.cu), restated."""
    if accurate:
        return "f32"
    tc_off = os.environ.get("MRB_POLICY_TC", "")[:1] == "0"
    if shape["H"] == 128 and shape["use_rnn"] and shape["A"] <= 8 and not tc_off:
        return "tc2"
    return "mma"


def random_model(shape, seed):
    """Random weights scaled by 1 / sqrt(fan_in), in state_dict layout."""
    rng = np.random.RandomState(seed)
    H, A, N = shape["H"], shape["A"], shape["N"]
    Din = shape["D"] + (N if shape["agent_id"] else 0)
    shapes = {"fc1.weight": (H, Din), "fc1.bias": (H,)}
    if shape["use_rnn"]:
        shapes.update({"rnn.weight_ih": (3 * H, H), "rnn.weight_hh": (3 * H, H), "rnn.bias_ih": (3 * H,), "rnn.bias_hh": (3 * H,)})
    else:
        shapes.update({"rnn.weight": (H, H), "rnn.bias": (H,)})
    shapes.update({"fc2.weight": (A, H), "fc2.bias": (A,)})
    fan_in = {"fc1": Din, "rnn": H, "fc2": H}
    prefixes = ["agents.%d." % i for i in range(N)] if shape["non_shared"] else [""]
    return {p + k: (rng.standard_normal(s) / np.sqrt(fan_in[k.split(".")[0]])).astype(np.float32)
            for p in prefixes for k, s in shapes.items()}


def make_policy(sd, shape, accurate):
    from marbler_b200.policy import Policy
    return Policy(sd, shape["N"], shape["D"], obs_agent_id=shape["agent_id"], device="cuda:0", accurate=accurate)


def assert_ran_on(kernel, fn):
    names = kernels_launched(fn, "policy_act")
    assert len(names) == 1 and KERNEL_NAME[kernel] in names[0], (kernel, names)


def q_bar(kernel, scale):
    rel, floor = Q_MAX[kernel]
    return rel * scale + floor


class Errors(object):
    """Checks one launch against the reference evaluated from the same input hidden state, and keeps the worst and
    median |q - q_ref| / |q_ref|max and the worst |h - h_ref| / max(1, |h_ref|max) over a case.

    The median is taken against the whole reference.  The max bar applies to q against fc2 of the kernel's own h'
    (`q_fc2`): an FP16 rounding of a large h' element that falls the other way in float64 moves q by up to half an FP16
    ulp of that element times its fc2 weight (measured 7e-4 for a Linear+ReLU model with |q|max 2.4), which says
    nothing about the kernel; h' itself is held to the h bar against the whole reference."""

    def __init__(self, kernel):
        self.kernel, self.q_max, self.q_meds, self.h_max = kernel, 0.0, [], 0.0

    def add(self, q, q_ref, h, h_ref, q_fc2):
        scale = float(q_ref.abs().max())
        worst = float((q.double() - q_fc2).abs().max())
        assert worst < q_bar(self.kernel, scale), (worst, scale)
        self.q_max = max(self.q_max, worst / scale)
        self.q_meds.append(float((q.double() - q_ref).abs().median()) / scale)
        self.h_max = max(self.h_max, float((h.double() - h_ref).abs().max()) / max(1.0, float(h_ref.abs().max())))
        return scale

    def check(self, what):
        q_med = float(np.median(self.q_meds))
        print("%s on %s: max |q - fc2_64(h')| = %.2e, median |q - q64| = %.2e (|q|max); max |h - h64| = %.2e"
              % (what, self.kernel, self.q_max, q_med, self.h_max))
        assert q_med < Q_MED[self.kernel], (what, q_med)
        assert self.h_max < H_MAX[self.kernel], (what, self.h_max)


def check_actions(kernel, a, q, q_ref, q_fc2):
    """The kernel's action is the first maximum of its own q (np.argmax); it is fc2_64's wherever that one's top-2 gap
    is wider than twice the max bar, and the whole reference's wherever its gap is wider than twice
    tests/test_policy.py's FP16 bar (1e-4 |q|max + 2e-4)."""
    an = a.cpu().numpy()
    assert np.array_equal(an, q.cpu().numpy().argmax(axis=-1))
    scale = float(q_ref.abs().max())
    for ref, gap in ((q_fc2, 2 * q_bar(kernel, scale)), (q_ref, 2 * (1e-4 * scale + 2e-4))):
        if ref.shape[-1] > 1:
            top = torch.sort(ref, dim=-1).values
            clear = ((top[..., -1] - top[..., -2]) > gap).cpu().numpy()
        else:
            clear = np.ones(an.shape, dtype=bool)
        assert np.array_equal(an[clear], ref.argmax(dim=-1).cpu().numpy()[clear])


# ------------------------------------------------------------------------------------------------ shape sweep

def S(H, use_rnn, D, agent_id, N, A, non_shared):
    return dict(H=H, use_rnn=use_rnn, D=D, agent_id=agent_id, N=N, A=A, non_shared=non_shared)


# (kernel it is meant to reach, accurate, shape); Din = D (+ N with the one-hot id)
CASES = [
    # tcgen05: dp 16 / 32 / 48 / 64 (weight ring 3, 3, 2, 2), A 1 / 5 / 8, shared and per-agent, N 1 .. 32
    ("tc2", False, S(128, True, 1, False, 1, 5, False)),        # Din 1
    ("tc2", False, S(128, True, 16, False, 4, 8, False)),       # Din 16
    ("tc2", False, S(128, True, 14, True, 3, 1, True)),         # Din 17
    ("tc2", False, S(128, True, 28, True, 5, 5, True)),         # Din 33
    ("tc2", False, S(128, True, 41, True, 7, 8, False)),        # Din 48
    ("tc2", False, S(128, True, 32, True, 32, 8, True)),        # Din 64
    ("tc2", False, S(128, True, 64, False, 3, 5, True)),        # Din 64, no id
    # mma.sync: hidden 64 GRU / Linear, hidden 128 Linear, hidden 128 GRU with 9 and 24 actions
    ("mma", False, S(64, True, 1, False, 2, 1, False)),         # Din 1
    ("mma", False, S(64, True, 45, True, 4, 9, True)),          # Din 49
    ("mma", False, S(64, False, 16, False, 3, 16, True)),       # Din 16
    ("mma", False, S(64, False, 60, True, 4, 24, False)),       # Din 64
    ("mma", False, S(128, False, 49, False, 2, 24, False)),     # Din 49
    ("mma", False, S(128, False, 1, False, 3, 1, True)),        # Din 1
    ("mma", False, S(128, True, 61, True, 3, 9, True)),         # Din 64
    ("mma", False, S(128, True, 12, True, 4, 24, False)),       # Din 16
    ("mma", False, S(128, True, 16, False, 5, 16, True)),       # Din 16
    # float32: hidden 64 / 128 x GRU / Linear, Din 1 and 64, A 1 and 24, shared and per-agent
    ("f32", True, S(64, True, 1, False, 2, 1, False)),
    ("f32", True, S(64, False, 60, True, 4, 24, True)),
    ("f32", True, S(128, True, 64, False, 3, 24, True)),
    ("f32", True, S(128, True, 1, False, 4, 1, False)),
    ("f32", True, S(128, False, 1, False, 2, 24, True)),
    ("f32", True, S(128, False, 61, True, 3, 1, False)),
]


def _case_id(c):
    k, _, s = c
    return "%s-H%d-%s-Din%d-N%d-A%d-%s" % (k, s["H"], "gru" if s["use_rnn"] else "lin", s["D"] + (s["N"] if s["agent_id"] else 0),
                                         s["N"], s["A"], "ns" if s["non_shared"] else "sh")


SENTINEL_H, SENTINEL_Q, SENTINEL_A = 1234.5, -999.0, -7


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_kernel_matches_float64_reference(case):
    """3 recurrent steps from a random hidden state, `fresh` on every 5th env from the second step, at batch sizes
    around the CTA edges (64 envs for mma.sync, 128 for tcgen05, 16 for float32).  Each launch covers the first B
    envs of larger buffers whose later rows must stay untouched; observation rows past B are NaN.  Each step is
    compared with the reference evaluated from the kernel's own input hidden state, so that an FP16 rounding that
    falls the other way in one step is not carried into the next."""
    kernel, accurate, shape = case
    routed = expected_kernel(shape, accurate)           # the MRB_POLICY_TC=0 rerun below sends the tc2 cases to mma.sync
    assert routed == kernel or (kernel, routed) == ("tc2", "mma")
    kernel = routed
    N, D, H, A = shape["N"], shape["D"], shape["H"], shape["A"]
    sd = random_model(shape, seed=11)
    pol = make_policy(sd, shape, accurate)
    dev = torch.device("cuda:0")
    batches = [1, 63, 64, 65, 127, 128, 129] + ([16, 17] if kernel == "f32" else [])
    Bmax, Bbuf, T = max(batches), max(batches) + 7, 3
    g = torch.Generator(device=dev).manual_seed(7)
    obs = [torch.randn((Bbuf, N, D), generator=g, device=dev) for _ in range(T)]
    for o in obs:
        o[Bmax:] = float("nan")
    h0 = torch.rand((Bbuf, N, H), generator=g, device=dev) * 2 - 1
    fresh = [None] + [(torch.arange(Bbuf, device=dev) % 5 == 2 + t).to(torch.uint8) for t in range(1, T)]
    err = Errors(kernel)
    for B in batches:
        hid = torch.full((Bbuf, N, H), SENTINEL_H, device=dev)
        hid[:B] = h0[:B]
        q = torch.full((Bbuf, N, A), SENTINEL_Q, device=dev)
        act = torch.full((Bbuf, N), SENTINEL_A, dtype=torch.int32, device=dev)
        for t in range(T):
            h_in = hid[:B].clone()
            run = lambda: pol.act(obs[t][:B], hid[:B], actions=act[:B], q=q[:B],
                                  fresh=None if fresh[t] is None else fresh[t][:B])
            if B == Bmax and t == 0:
                assert_ran_on(kernel, run)
            else:
                run()
            torch.cuda.synchronize()
            q_ref, h_ref = step64(sd, shape, obs[t][:B], h_in, None if fresh[t] is None else fresh[t][:B].bool(),
                                  fp16=not accurate)
            q_fc2 = fc2_64(sd, shape, hid[:B], fp16=not accurate)
            check_actions(kernel, act[:B], q[:B], q_ref, q_fc2)
            err.add(q[:B], q_ref, hid[:B], h_ref, q_fc2)
        assert bool((hid[B:] == SENTINEL_H).all()) and bool((q[B:] == SENTINEL_Q).all()) and bool((act[B:] == SENTINEL_A).all()), B
    err.check(_case_id(case) + " (B %s)" % ",".join(map(str, batches)))


@pytest.mark.gpu
def test_tc2_shapes_on_the_mma_sync_kernel():
    """MRB_POLICY_TC=0 sends the tcgen05 shapes to the mma.sync kernel, which must meet the same bars and tie rule.
    The switch is read once per process, hence the subprocess."""
    env = dict(os.environ, MRB_POLICY_TC="0")
    res = subprocess.run([sys.executable, "-m", "pytest", __file__, "-q", "-s", "-m", "gpu", "-p", "no:cacheprovider",
                          "-k", "test_kernel_matches_float64_reference and tc2 or test_ties_go_to_the_lowest_index and tc2"],
                         env=env, capture_output=True, text=True, timeout=900)
    print(res.stdout[-6000:])
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "passed" in res.stdout and " on mma:" in res.stdout and " on tc2:" not in res.stdout


# ------------------------------------------------------------------------------------------------ persistent steady state

def _chunks(B, N):
    """128-aligned chunks of (num_sms // N) * 128 envs: one tile per CTA of the persistent kernel."""
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    step = (num_sms // N) * 128
    return [(lo, min(B, lo + step)) for lo in range(0, B, step)]


def _tiles_per_cta(B, N):
    """(grid, tiles, tiles per CTA) of a persistent tcgen05 launch over B envs, as mrb_policy_act sizes it."""
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = (B + 127) // 128 * N
    grid = min(num_sms // N * N, tiles)
    return grid, tiles, -(-tiles // grid)


PERSISTENT = [
    ("pcp-shipped-N4", dict(H=128, use_rnn=True, D=16, agent_id=True, N=4, A=5, non_shared=False), 65536),
    ("per-agent-N3", dict(H=128, use_rnn=True, D=20, agent_id=False, N=3, A=5, non_shared=True), 30000),
    ("per-agent-N5", dict(H=128, use_rnn=True, D=11, agent_id=True, N=5, A=8, non_shared=True), 30000),
    ("per-agent-N7", dict(H=128, use_rnn=True, D=30, agent_id=True, N=7, A=6, non_shared=True), 30000),
    ("per-agent-N32", dict(H=128, use_rnn=True, D=20, agent_id=False, N=32, A=5, non_shared=True), 2510),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,shape,B", PERSISTENT, ids=[p[0] for p in PERSISTENT])
def test_persistent_tc2_launch_equals_one_tile_per_cta_launches(name, shape, B):
    """A row's arithmetic does not depend on which CTA or which tile iteration handles it, so one launch in which
    every CTA loops over many tiles (second use of each activation buffer, reuse of both TMEM halves, the weight ring
    running on across tiles, the head loaded once per CTA) must equal, bit for bit, launches over chunks in which each
    CTA gets one tile.  3 recurrent steps, `fresh` on every 7th env; the full launch also meets the float64 bars."""
    N, D, H, A = shape["N"], shape["D"], shape["H"], shape["A"]
    assert expected_kernel(shape, False) == "tc2"
    if name.startswith("pcp"):
        z, sd, fshape = _fixture("PredatorCapturePrey_vdn")
        assert all(fshape[k] == shape[k] for k in fshape)
    else:
        sd = random_model(shape, seed=23)
    pol = make_policy(sd, shape, False)
    dev = torch.device("cuda:0")
    grid, tiles, per_cta = _tiles_per_cta(B, N)
    chunks = _chunks(B, N)
    assert grid % N == 0 and all(_tiles_per_cta(hi - lo, N)[2] == 1 for lo, hi in chunks)
    assert per_cta >= (10 if name.startswith("pcp") else 4), per_cta
    assert name.startswith("pcp") or B % 128 != 0               # a ragged last tile
    print("%s: %d envs, grid %d, %d tiles, %d tiles per CTA (one-tile chunks: %d)" % (name, B, grid, tiles, per_cta, len(chunks)))
    g = torch.Generator(device=dev).manual_seed(5)
    h0 = torch.rand((B, N, H), generator=g, device=dev) * 2 - 1
    hid1, hid2 = h0.clone(), h0.clone()
    q1, q2 = torch.empty((B, N, A), device=dev), torch.empty((B, N, A), device=dev)
    a1, a2 = torch.empty((B, N), dtype=torch.int32, device=dev), torch.empty((B, N), dtype=torch.int32, device=dev)
    err = Errors("tc2")
    for t in range(3):
        obs = torch.rand((B, N, D), generator=g, device=dev) * 3 - 1.5
        h_in = hid1.clone()
        fresh = ((torch.arange(B, device=dev) + t) % 7 == 0).to(torch.uint8)
        pol.act(obs, hid1, actions=a1, q=q1, fresh=fresh)
        for lo, hi in chunks:
            pol.act(obs[lo:hi], hid2[lo:hi], actions=a2[lo:hi], q=q2[lo:hi], fresh=fresh[lo:hi])
        torch.cuda.synchronize()
        assert torch.equal(q1, q2) and torch.equal(hid1, hid2) and torch.equal(a1, a2), t
        q_ref, h_ref = step64(sd, shape, obs, h_in, fresh.bool(), fp16=True)
        q_fc2 = fc2_64(sd, shape, hid1, fp16=True)
        check_actions("tc2", a1, q1, q_ref, q_fc2)
        err.add(q1, q_ref, hid1, h_ref, q_fc2)
        del q_ref, h_ref, h_in, q_fc2
    err.check("%s, %d tiles per CTA" % (name, per_cta))


@pytest.mark.gpu
def test_closed_loop_at_production_size_equals_chunked_launches():
    """Rollout on 65,536 PredatorCapturePrey envs with the shipped checkpoint, CUDA graphs of 8 steps: 20 steps run as
    one eager warm-up, two graph replays and an eager tail of 3.  A second VecEnv with the same seed, driven by hand
    with the policy applied over one-tile-per-CTA chunks, must end in the same state bit for bit."""
    from marbler_b200.policy import Rollout
    from marbler_b200.vec_env import VecEnv
    z, sd, shape = _fixture("PredatorCapturePrey_vdn")
    cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    B, T = 65536, 20
    pol = make_policy(sd, shape, False)
    assert _tiles_per_cta(B, shape["N"])[2] > 10
    ro = Rollout(VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=21, auto_reset=True), pol,
                 use_graph=True, steps_per_graph=8)
    ro.reset()
    ro.run(T)
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=21, auto_reset=True)
    env.reset()
    env.done.fill_(1)
    hidden = pol.init_hidden(B)
    actions = torch.zeros((B, shape["N"]), dtype=torch.int32, device="cuda:0")
    for _ in range(T):
        for lo, hi in _chunks(B, shape["N"]):
            pol.act(env.obs[lo:hi], hidden[lo:hi], actions=actions[lo:hi], fresh=env.done[lo:hi])
        env.step(actions)
    torch.cuda.synchronize()
    assert ro._graph is not None
    for a, b, what in ((ro.env.state_f64, env.state_f64, "state_f64"), (ro.env.state_i32, env.state_i32, "state_i32"),
                       (ro.hidden, hidden, "hidden"), (ro.actions, actions, "actions"), (ro.env.obs, env.obs, "obs")):
        assert torch.equal(a, b), what


# ------------------------------------------------------------------------------------------------ ties and alignment

TIES = [  # (kernel, accurate, shape, tied action sets): mma.sync columns c sit in tile c // 8, lane quad (c % 8) // 2
    ("tc2", False, S(128, True, 16, True, 4, 8, False), [(1, 6), (3, 4), (5, 7), tuple(range(8))]),
    ("mma", False, S(128, True, 16, True, 4, 24, False), [(2, 10), (7, 8), (6, 9, 17), (5, 12, 23), tuple(range(24))]),
    ("mma", False, S(64, False, 16, False, 3, 24, True), [(2, 10), (7, 8), tuple(range(24))]),
    ("f32", True, S(128, True, 16, True, 4, 24, False), [(2, 10), (7, 8), (6, 9, 17), tuple(range(24))]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", TIES, ids=[_case_id(c[:3]) for c in TIES])
def test_ties_go_to_the_lowest_index(case):
    """fc2 rows and biases duplicated, the duplicates lifted above every other action: q ties exactly, and the action
    is the lowest tied index, as np.argmax returns (utilities/misc.py:170)."""
    kernel, accurate, shape, tie_sets = case
    kernel = expected_kernel(shape, accurate)
    N, D, A = shape["N"], shape["D"], shape["A"]
    B = 200
    g = torch.Generator(device="cuda:0").manual_seed(9)
    obs = torch.randn((B, N, D), generator=g, device="cuda:0")
    for tied in tie_sets:
        sd = random_model(shape, seed=31)
        for p in (["agents.%d." % i for i in range(N)] if shape["non_shared"] else [""]):
            w, b = sd[p + "fc2.weight"], sd[p + "fc2.bias"]
            for c in tied:
                w[c], b[c] = w[tied[-1]], b[tied[-1]] + (0 if len(tied) == A else 20)
        pol = make_policy(sd, shape, accurate)
        hid = torch.rand((B, N, shape["H"]), generator=g, device="cuda:0") - 0.5
        q = torch.zeros((B, N, A), device="cuda:0")
        act = pol.act(obs, hid, q=q)
        torch.cuda.synchronize()
        qt = q[..., list(tied)]
        assert bool((qt == qt[..., :1]).all()), (kernel, tied)
        assert bool((q.max(dim=-1).values == qt[..., 0]).all()), (kernel, tied)
        assert bool((act == min(tied)).all()), (kernel, tied, torch.unique(act).tolist())


ALIGN = [("tc2", False, S(128, True, 16, True, 4, 5, False)), ("mma", False, S(64, True, 30, False, 4, 5, True)),
         ("f32", True, S(128, True, 16, True, 4, 5, False))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ALIGN, ids=[_case_id(c) for c in ALIGN])
def test_hidden_must_be_16_byte_aligned(case):
    """The kernels move hidden rows as float4 / float2: a contiguous view 2 floats into an allocation passes every
    shape check but is only 8-byte aligned, and mrb_policy_act refuses it on every path before any launch.  A view 4
    floats in is 16-byte aligned and gives exactly what an aligned copy gives."""
    kernel, accurate, shape = case
    N, D, H, A = shape["N"], shape["D"], shape["H"], shape["A"]
    B = 300
    pol = make_policy(random_model(shape, seed=3), shape, accurate)
    g = torch.Generator(device="cuda:0").manual_seed(4)
    obs = torch.randn((B, N, D), generator=g, device="cuda:0")
    h0 = torch.rand((B, N, H), generator=g, device="cuda:0") - 0.5
    n = B * N * H
    bad = torch.empty(n + 2, device="cuda:0")[2:].view(B, N, H)
    assert bad.is_contiguous() and bad.data_ptr() % 16 == 8
    bad.copy_(h0)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        pol.act(obs, bad)
    torch.cuda.synchronize()
    assert torch.equal(bad, h0)
    off = torch.empty(n + 4, device="cuda:0")[4:].view(B, N, H)
    assert off.data_ptr() % 16 == 0 and off.data_ptr() % 256 != 0
    off.copy_(h0)
    ref = h0.clone()
    q1, q2 = torch.zeros((B, N, A), device="cuda:0"), torch.zeros((B, N, A), device="cuda:0")
    assert expected_kernel(shape, accurate) == kernel
    a1, a2 = pol.act(obs, off, q=q1), pol.act(obs, ref, q=q2)
    torch.cuda.synchronize()
    assert torch.equal(off, ref) and torch.equal(q1, q2) and torch.equal(a1, a2)
