"""What Rollout(skip_finished=True) saves (mrb_step_masked), measured in one process with the variants alternated:

  * the wall time of Rollout.collect() (episode_limit T) and Rollout.evaluate() (K episodes per env) with skip_finished
    off and on, for three workloads: PredatorCapturePrey with 4 robots at 65,536 envs and the shipped vdn checkpoint;
    PredatorCapturePrey with 20 robots in bench.py's configuration (131,072 envs, random-init policy); MaterialTransport
    at 262,144 envs with the shipped mappo_ns checkpoint (softmax);
  * the fraction of env steps skipped, from the env_steps counter of env.stats (on against off);
  * the step call alone, from CUDA-graph replays: mrb_step, mrb_step_masked with an all-ones mask, and mrb_step_masked
    with an all-zeros mask (the compaction and an empty step launch: the fixed cost of the masked call).

Usage: python scripts/skip_time.py [--out FILE.json] [--rounds R]   (prints the JSON either way; needs a B200)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import golden_util as gu  # noqa: E402
from marbler_b200 import config  # noqa: E402
from marbler_b200.policy import EpisodeBatch, EvalLog, Exploration, Policy, Rollout  # noqa: E402
from marbler_b200.vec_env import VecEnv  # noqa: E402

PCP20 = dict(predator=10, capture=10, ROBOT_INIT_RIGHT_THRESH=0.1, num_neighbors=3)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "not read", "sm_max_clock": "not read"}


def stats(x):
    return {"median": float(np.median(x)), "min": float(min(x)), "max": float(max(x))}


def checkpoint(name):
    z = np.load(os.path.join(gu.GOLDEN, "policy", name + ".npz"))
    return {k[3:]: z[k] for k in z.files if k.startswith("sd.")}


def random_agent(N, D, A, H=128):
    g = torch.Generator().manual_seed(0)
    u = lambda *shape: (torch.rand(shape, generator=g) * 2 - 1) / (shape[-1] ** 0.5)
    return {"fc1.weight": u(H, D + N), "fc1.bias": u(H), "rnn.weight_ih": u(3 * H, H), "rnn.weight_hh": u(3 * H, H),
            "rnn.bias_ih": u(3 * H), "rnn.bias_hh": u(3 * H), "fc2.weight": u(A, H), "fc2.bias": u(A)}


# name: (scenario, config, envs, checkpoint or None (random init), exploration mode, K)
CASES = {
    "PCP4_65536_vdn": ("PredatorCapturePrey", dict(gu.Golden("PredatorCapturePrey_rollout").cfg), 65536,
                       "PredatorCapturePrey_vdn", "epsilon_greedy", 10),
    "PCP20_131072_random": ("PredatorCapturePrey", dict(config.load_yaml(config.default_config_path("PredatorCapturePrey")),
                                                        **PCP20), 131072, None, "epsilon_greedy", 2),
    "MaterialTransport_262144_mappo_ns": ("MaterialTransport",
                                          config.load_yaml(config.default_config_path("MaterialTransport")), 262144,
                                          "MaterialTransport_mappo_ns", "softmax", 10),
}


def make(case, skip):
    scenario, cfg, B, ck, mode, K = CASES[case]
    env = VecEnv(scenario, cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
    T = env.c.max_episode_steps + 1
    sd = checkpoint(ck) if ck else random_agent(env.N, env.D, env.n_actions)
    ex = Exploration(mode, seed=1, eps_start=0.05, eps_finish=0.05, device="cuda:0")
    return Rollout(env, Policy(sd, env.N, env.D, device="cuda:0"), use_graph=True, steps_per_graph=16, explore=ex,
                   record=EpisodeBatch(env, T), evaluate=EvalLog(env, K), skip_finished=skip)


def timed(ro, fn):
    ro.env.stats.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, float(ro.env.stats[6].item())       # MRB_STAT_ENV_STEPS


def step_calls(env, reps=20, per_graph=16):
    """ms per call of mrb_step, and of mrb_step_masked with all-ones and all-zeros masks, from graph replays
    alternated over `reps` rounds."""
    actions = torch.full((env.B, env.N), 4, dtype=torch.int32, device="cuda:0")
    ones = torch.ones(env.B, dtype=torch.uint8, device="cuda:0")
    zeros = torch.zeros(env.B, dtype=torch.uint8, device="cuda:0")
    variants = {"mrb_step": None, "masked_all_ones": ones, "masked_all_zeros": zeros}
    graphs = {}
    env.reset()
    for name, m in variants.items():
        env.step(actions, active=m)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(per_graph):
                env.step(actions, active=m)
        graphs[name] = g
    out = {k: [] for k in variants}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for name, g in graphs.items():
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            out[name].append(e0.elapsed_time(e1) / per_graph)
    return {k: stats(v) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cases", default=",".join(CASES))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "rounds": args.rounds, "cases": {}}
    for case in args.cases.split(","):
        rounds = max(1, args.rounds // 2) if "PCP20" in case else args.rounds        # 53 ms per env step
        ros = {s: make(case, s) for s in (False, True)}
        # warm-up: capture the graphs; every env then has its K episodes.  The first collect() starts from the same state
        # in both variants, so its batches are equal; after it the skipped envs' episode counters (which key the reset
        # streams) lag behind, so later calls reset into other episodes
        first = [ro.collect() for ro in ros.values()]
        assert all(torch.equal(first[0][f], first[1][f]) for f in first[0]), case
        for ro in ros.values():
            ro.evaluate()
        torch.cuda.synchronize()
        wall = {(w, s): [] for w in ("collect", "evaluate") for s in (False, True)}
        steps = {}
        for _ in range(rounds):
            for w in ("collect", "evaluate"):
                for s, ro in ros.items():
                    ms, n = timed(ro, ro.collect if w == "collect" else ro.evaluate)
                    wall[(w, s)].append(ms)
                    steps[(w, s)] = n
        env = ros[False].env
        T, K = env.c.max_episode_steps + 1, ros[False].eval_log.episodes
        r = {"envs": env.B, "agents": env.N, "T": T, "K": K, "rounds": rounds}
        for w in ("collect", "evaluate"):
            off, on = np.median(wall[(w, False)]), np.median(wall[(w, True)])
            r[w] = {"wall_ms_off": stats(wall[(w, False)]), "wall_ms_on": stats(wall[(w, True)]),
                    "env_steps_off": steps[(w, False)], "env_steps_on": steps[(w, True)],
                    "skipped_fraction": 1.0 - steps[(w, True)] / steps[(w, False)],
                    "time_saved_fraction": 1.0 - on / off}
        del ros
        torch.cuda.empty_cache()
        scenario, cfg, B = CASES[case][:3]
        r["step_call_ms"] = step_calls(VecEnv(scenario, cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True),
                                       reps=5 if "PCP20" in case else 20, per_graph=4 if "PCP20" in case else 16)
        res["cases"][case] = r
        torch.cuda.empty_cache()
    res["note"] = ("wall: host clock around Rollout.collect() / evaluate() (begin, reset, T or K * T env steps from graph "
                   "replays of 16 steps) and a synchronise; the first collect() of the two variants is checked equal. "
                   "skipped_fraction: 1 - env_steps(on) / env_steps(off) from env.stats. step_call_ms: graph replays of "
                   "the step call alone; masked_all_zeros is the compaction plus a step launch whose items all exit")
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
