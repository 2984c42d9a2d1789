"""Cost of exploratory action selection (mrb_select_actions), measured in one process with the variants alternated:

  * the closed loop (policy -> [selection] -> step, CUDA-graph replays of 16 env steps) on 65,536 PredatorCapturePrey
    envs with the shipped hidden-128 GRU checkpoint: greedy, epsilon-greedy (eps 0.05, EPyMARL's flat value) and
    softmax, as time per env step;
  * one selection call alone (selection kernel + counter advance, from a graph of 100 calls) against the HBM floor of
    the selection kernel (epsilon-greedy 4 B in + 4 B out per agent, softmax 4 A B of q in + 4 B out), and the
    selection kernel's own duration from a profiler pass;
  * the policy kernel with and without the q output for the three shipped checkpoint shapes (262,144 agents).

Usage: python scripts/explore_time.py [--out FILE.json]   (prints the JSON either way; needs a B200)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import golden_util as gu  # noqa: E402
from marbler_b200.policy import Exploration, Policy, Rollout  # noqa: E402
from marbler_b200.vec_env import VecEnv  # noqa: E402

B, N = 65536, 4
HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "not read", "sm_max_clock": "not read"}


def checkpoint(name):
    z = np.load(os.path.join(gu.GOLDEN, "policy", name + ".npz"))
    return {k[3:]: z[k] for k in z.files if k.startswith("sd.")}


def elapsed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def explorer(mode):
    return None if mode == "greedy" else Exploration(mode, seed=1, eps_start=0.05, eps_finish=0.05, device="cuda:0")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    modes = ("greedy", "epsilon_greedy", "softmax")
    cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    sd = checkpoint("PredatorCapturePrey_vdn")

    # ---- closed loop
    loops = {}
    for m in modes:
        env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
        ro = Rollout(env, Policy(sd, N, 16, device="cuda:0"), use_graph=True, steps_per_graph=16, explore=explorer(m))
        ro.reset()
        ro.run(33)
        loops[m] = ro
    torch.cuda.synchronize()
    closed = {m: [] for m in modes}
    for _ in range(args.rounds):
        for m in modes:
            closed[m].append(elapsed(lambda: loops[m].run(16), 20) / 16)
    del loops

    # ---- one selection call alone
    actions = torch.zeros((B, N), dtype=torch.int32, device="cuda:0")
    q = torch.randn((B, N, 5), device="cuda:0")
    sel = {}
    for m in ("epsilon_greedy", "softmax"):
        ex = explorer(m)
        call = (lambda ex=ex: ex.select(actions, q))
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(100):
                call()
        sel[m] = (g, call)
    select_ms = {m: [] for m in sel}
    for _ in range(args.rounds):
        for m, (g, _) in sel.items():
            select_ms[m].append(elapsed(g.replay, 10) / 100)
    kernel_us = {}
    from torch.profiler import ProfilerActivity, profile
    for m, (_, call) in sel.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(200):
                call()
            torch.cuda.synchronize()
        d = [e.device_time for e in prof.events() if "select_actions_kernel" in e.name]
        kernel_us[m] = float(np.median(d)) if d else None
    floor_bytes = {"epsilon_greedy": B * N * 8, "softmax": B * N * (4 * 5 + 4)}

    # ---- the policy kernel with and without the q output, shipped shapes
    pol_ms = {}
    for name, D in (("PredatorCapturePrey_vdn", 16), ("ArcticTransport_qmix_ns", 30), ("MaterialTransport_mappo_ns", 9)):
        pol = Policy(checkpoint(name), N, D, device="cuda:0")
        obs = torch.rand((B, N, D), device="cuda:0") * 2 - 1
        hid = pol.init_hidden(B)
        act = torch.zeros((B, N), dtype=torch.int32, device="cuda:0")
        qo = torch.zeros((B, N, pol.n_actions), device="cuda:0")
        variants = {"no_q": lambda: pol.act(obs, hid, actions=act), "q": lambda: pol.act(obs, hid, actions=act, q=qo)}
        for f in variants.values():
            for _ in range(5):
                f()
        torch.cuda.synchronize()
        res = {k: [] for k in variants}
        for _ in range(args.rounds):
            for k, f in variants.items():
                res[k].append(elapsed(f, 50))
        pol_ms[name] = {"n_actions": pol.n_actions, "hidden": pol.hidden_dim,
                        "ms_without_q": float(np.median(res["no_q"])), "ms_with_q": float(np.median(res["q"])),
                        "spread_without_q": [float(min(res["no_q"])), float(max(res["no_q"]))],
                        "spread_with_q": [float(min(res["q"])), float(max(res["q"]))]}

    med = {m: float(np.median(v)) for m, v in closed.items()}
    out = {
        "card": card(), "envs": B, "agents": B * N, "rounds": args.rounds,
        "closed_loop_ms_per_env_step": {m: {"median": med[m], "min": float(min(closed[m])), "max": float(max(closed[m]))}
                                        for m in modes},
        "closed_loop_vs_greedy": {m: med[m] / med["greedy"] - 1.0 for m in modes},
        "closed_loop_note": "PredatorCapturePrey_vdn checkpoint (hidden 128 GRU, tcgen05 kernel); epsilon 0.05 flat; "
                            "softmax reads the q the policy kernel then writes; 16 env steps per graph",
        "selection_call_us": {m: float(np.median(v)) * 1e3 for m, v in select_ms.items()},
        "selection_kernel_us_profiler": kernel_us,
        "selection_hbm_floor_us": {m: b / (HBM_TBPS * 1e12) * 1e6 for m, b in floor_bytes.items()},
        "selection_note": "a call = selection kernel + one-thread counter advance, from a CUDA graph of 100 calls; "
                          "softmax over 5 actions; floor at %.1f TB/s" % HBM_TBPS,
        "policy_kernel": pol_ms,
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
