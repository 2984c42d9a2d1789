"""Cost of loading new weights into a policy (Policy.load_state_dict -> mrb_policy_load), against the rebuild it
replaces, measured in one process:

  * the load_state_dict call from device tensors (the learner's parameters): CUDA events around each call, median
    over `--calls` warm calls, and the pack kernel alone from a torch.profiler pass, against its HBM floor (the
    weights read once plus every image word written, at the data sheet's 7.7 TB/s);
  * the rebuild path: state_dict().cpu(), Policy(...), Rollout(...) and its first collect() with the graph capture,
    minus a plain collect() on the rebuilt rollout (host clock, each end synchronised; median of `--rounds`);
  * mrb_policy_create from host weights (host clock, synchronous call), for this library and, with --parent-lib,
    another build of it (the C signature is the same across ABI versions).

Models: the three shipped checkpoints in their scenarios and a 32-agent per-agent hidden-128 GRU on a 32-robot
PredatorCapturePrey team (random weights).  Collections are epsilon-greedy with recording, as a training loop runs them.

Usage: python scripts/policy_load_time.py [--out FILE.json] [--parent-lib PATH]   (prints the JSON; needs a B200)."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import golden_util as gu  # noqa: E402
from marbler_b200 import _lib, config  # noqa: E402
from marbler_b200.policy import EpisodeBatch, Exploration, Policy, Rollout, flatten_state_dict  # noqa: E402
from marbler_b200.vec_env import VecEnv  # noqa: E402

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


def per_agent_gru(N, D, A, H=128, seed=0):
    rng = np.random.RandomState(seed)
    w = lambda *s: (rng.standard_normal(s) / np.sqrt(s[-1])).astype(np.float32)
    one = {"fc1.weight": (H, D), "fc1.bias": (H,), "rnn.weight_ih": (3 * H, H), "rnn.weight_hh": (3 * H, H),
           "rnn.bias_ih": (3 * H,), "rnn.bias_hh": (3 * H,), "fc2.weight": (A, H), "fc2.bias": (A,)}
    return {"agents.%d.%s" % (i, k): w(*s) for i in range(N) for k, s in one.items()}


def models():
    """(name, scenario, config, envs, episode limit, state_dict)"""
    out = []
    for scen, ck in (("PredatorCapturePrey", "PredatorCapturePrey_vdn"), ("ArcticTransport", "ArcticTransport_qmix_ns"),
                     ("MaterialTransport", "MaterialTransport_mappo_ns")):
        cfg = config.load_yaml(config.default_config_path(scen))
        cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg) if scen == "PredatorCapturePrey" else cfg
        out.append((ck, scen, cfg, 65536, 81, checkpoint(ck)))
    N = 32
    cfg = dict(config.load_yaml(config.default_config_path("PredatorCapturePrey")), predator=N // 2, capture=N - N // 2,
               ROBOT_INIT_RIGHT_THRESH=0.1, start_dist=0.25)
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=1, device="cuda:0")
    out.append(("per_agent_gru_N32_H128", "PredatorCapturePrey", cfg, 4096, 81, per_agent_gru(N, env.D, env.n_actions)))
    return out


def image_words(pol, n_weights):
    """32-bit words the pack kernel writes (every image the policy holds), restated from csrc/policy.cu."""
    H, A, N = pol.hidden_dim, pol.n_actions, pol.n_agents
    Din = pol.obs_dim + (N if pol.obs_agent_id else 0)
    sets = N if pol.non_shared else 1
    KS1, NT, KS, AT, G = (Din + 15) // 16, H // 8, H // 16, (A + 7) // 8, 6 if pol.use_rnn else 1
    wpack = NT * KS1 * 64 + H + (6 * H if pol.use_rnn else H) + AT * KS * 64 + AT * 8 + NT * G * KS * 64
    dp = (Din + 15) & ~15
    tc2 = 0
    if not pol.accurate and H == 128 and pol.use_rnn and A <= 8:
        tc2 = 128 * (dp + 8) // 2 + (128 + 3 * 128 + 3 * 128 + 32) + A * 128 + 12 * 64 * 128 * 2 // 4
    return sets * (wpack + tc2)


def create_time(lib_path, pol, flat, reps=7):
    L = C.CDLL(lib_path)
    L.mrb_policy_create.argtypes = [C.POINTER(_lib.PolicyDesc), C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
    L.mrb_policy_destroy.argtypes = [C.c_void_p]
    Din = pol.obs_dim + (pol.n_agents if pol.obs_agent_id else 0)
    d = _lib.PolicyDesc(C.sizeof(_lib.PolicyDesc), pol.obs_dim, Din, pol.hidden_dim, pol.n_actions, pol.n_agents,
                        int(pol.obs_agent_id), int(pol.use_rnn), int(pol.non_shared), 0)
    ts = []
    for _ in range(reps + 1):
        h = C.c_void_p()
        t0 = time.perf_counter()
        rc = L.mrb_policy_create(C.byref(d), 0, flat.ctypes.data_as(C.c_void_p), flat.size, C.byref(h))
        ts.append((time.perf_counter() - t0) * 1e3)
        assert rc == 0, rc
        L.mrb_policy_destroy(h)
    return statistics.median(ts[1:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--parent-lib", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "hbm_tbps_datasheet": HBM_TBPS, "models": []}
    for name, scen, cfg, B, T, sd in models():
        env = VecEnv(scen, cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
        N, D = env.N, env.D
        flat, _ = flatten_state_dict(sd, N)
        learner = {k: torch.nn.Parameter(torch.as_tensor(v, device="cuda:0")) for k, v in sd.items()}
        pol = Policy(sd, N, D, device="cuda:0")
        ex = Exploration("epsilon_greedy", seed=1, eps_start=0.05, eps_finish=0.05, device="cuda:0")
        rec = EpisodeBatch(env, T)
        ro = Rollout(env, pol, use_graph=True, steps_per_graph=16, explore=ex, record=rec)
        ro.collect()
        torch.cuda.synchronize()

        # ---- load_state_dict, CUDA events around each call
        for _ in range(20):
            pol.load_state_dict(learner)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.calls)]
        host = []
        torch.cuda.synchronize()
        for e0, e1 in ev:
            e0.record()
            t0 = time.perf_counter()
            pol.load_state_dict(learner)
            host.append((time.perf_counter() - t0) * 1e3)
            e1.record()
        torch.cuda.synchronize()
        load_ms = statistics.median(e0.elapsed_time(e1) for e0, e1 in ev)

        # ---- the pack kernel alone (profiler pass of its own)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(50):
                pol.load_state_dict(learner)
            torch.cuda.synchronize()
        kern = [e.device_time_total for e in prof.events() if "policy_pack_kernel" in e.name]
        other = sorted({e.name for e in prof.events() if "policy_pack_kernel" not in e.name and e.device_time_total > 0})
        kernel_us = statistics.median(kern) if kern else None
        nbytes = 4 * flat.size + 4 * image_words(pol, flat.size)
        floor_us = nbytes / (HBM_TBPS * 1e12) * 1e6

        # ---- rebuild path vs a plain collect
        rebuild, plain, load_collect = [], [], []
        for _ in range(args.rounds):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sd_cpu = {k: v.detach().cpu() for k, v in learner.items()}
            p2 = Policy(sd_cpu, N, D, device="cuda:0")
            r2 = Rollout(env, p2, use_graph=True, steps_per_graph=16, explore=ex, record=rec)
            r2.collect()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            r2.collect()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            ro.policy.load_state_dict(learner)
            ro.collect()
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            rebuild.append((t1 - t0) * 1e3)
            plain.append((t2 - t1) * 1e3)
            load_collect.append((t3 - t2) * 1e3)
            del r2, p2
        m = {"model": name, "scenario": scen, "envs": B, "episode_limit": T, "n_agents": N, "num_weights": int(flat.size),
             "weights_mb": 4 * flat.size / 1e6, "image_mb": 4 * image_words(pol, flat.size) / 1e6,
             "load_state_dict_ms_median_events": load_ms, "load_state_dict_host_ms_median": statistics.median(host),
             "calls_timed": args.calls, "pack_kernel_us_median_profiler": kernel_us,
             "other_kernels_in_load": other, "pack_hbm_floor_us": floor_us,
             "pack_kernel_over_floor": (kernel_us / floor_us) if kernel_us else None,
             "rebuild_then_collect_ms_median": statistics.median(rebuild), "plain_collect_ms_median": statistics.median(plain),
             "load_then_collect_ms_median": statistics.median(load_collect),
             "rebuild_minus_plain_collect_ms": statistics.median(rebuild) - statistics.median(plain),
             "load_share_of_plain_collect": load_ms / statistics.median(plain),
             "mrb_policy_create_ms": create_time(_lib.LIB_PATH, pol, flat)}
        if args.parent_lib:
            m["mrb_policy_create_ms_parent"] = create_time(args.parent_lib, pol, flat)
        res["models"].append(m)
        print(json.dumps(m), flush=True)
        del ro, pol, rec, env, learner
        torch.cuda.empty_cache()
    txt = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
