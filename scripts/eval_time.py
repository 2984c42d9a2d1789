"""Cost of on-device evaluation (mrb_eval_begin / mrb_eval_step, policy.EvalLog), measured in one process with the
variants alternated:

  * the closed loop (policy [-> selection] -> step [-> eval], CUDA-graph replays of 16 env steps) on 65,536
    PredatorCapturePrey envs with the shipped hidden-128 GRU checkpoint, greedy and epsilon-greedy, with and without
    evaluate=, as time per env step (each timed window of 80 steps starts with mrb_eval_begin; K = 10, so rows are
    written throughout);
  * the eval kernel alone (a graph of begin + 80 step calls over synthetic buffers in which about 2 % of the envs finish
    per step), against its HBM floor from the bytes the shapes imply, and the kernel's own duration from a profiler pass;
  * the wall time of Rollout.evaluate() with K = 10 (begin, reset, 10 * 81 env steps), and the fraction of those env
    steps taken by envs that had already logged their K episodes (from the table: K * 81 minus the sum of an env's
    K lengths);
  * an early exit that reads count.min() on the host every 80 steps and stops once every env has logged K episodes,
    against evaluate()'s fixed step count;
  * the bias of the windowed env statistics: K = 1 return_mean against the env.stats mean over the same 81 steps.

Usage: python scripts/eval_time.py [--out FILE.json]   (prints the JSON either way; needs a B200)."""
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
from marbler_b200.policy import EvalLog, Exploration, Policy, Rollout  # noqa: E402
from marbler_b200.vec_env import VecEnv  # noqa: E402

B, N, D, K = 65536, 4, 16, 10
HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "not read", "sm_max_clock": "not read"}


def elapsed(fn, reps=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def eval_bytes(done_fraction):
    """Bytes one mrb_eval_step moves per env: reads reward and dist (N floats each), done and the three accumulators,
    writes the accumulators back; an env that finishes also reads count, message and remaining and writes one row
    (return 8, length 4, message 1, timeout 1, remaining 4, dist 4) and count."""
    every = 4 * N + 4 * N + 1 + 2 * (8 + 4 + 8)
    finish = 4 + 1 + 4 + 22 + 4
    return every + done_fraction * finish


def make(cfg, sd, mode, evaluate, seed=3):
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=seed, auto_reset=True)
    ex = Exploration("epsilon_greedy", seed=1, eps_start=0.05, eps_finish=0.05, device="cuda:0") \
        if mode == "epsilon_greedy" else None
    return Rollout(env, Policy(sd, N, D, device="cuda:0"), use_graph=True, steps_per_graph=16, explore=ex,
                   evaluate=EvalLog(env, K) if evaluate else None)


def stats(x):
    return {"median": float(np.median(x)), "min": float(min(x)), "max": float(max(x))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    z = np.load(os.path.join(gu.GOLDEN, "policy", "PredatorCapturePrey_vdn.npz"))
    sd = {k[3:]: z[k] for k in z.files if k.startswith("sd.")}
    T = int(VecEnv("PredatorCapturePrey", cfg, num_envs=1, device="cuda:0").c.max_episode_steps) + 1

    # ---- closed loop, with and without evaluation, greedy and epsilon-greedy
    loops = {(m, e): make(cfg, sd, m, e) for m in ("greedy", "epsilon_greedy") for e in (False, True)}
    for ro in loops.values():
        ro.reset()
        ro.run(T)
    torch.cuda.synchronize()

    def window(ro):
        if ro.eval_log is not None:
            ro.eval_log.begin()
        for _ in range(5):
            ro.run(16)

    closed = {v: [] for v in loops}
    for _ in range(args.rounds):
        for v, ro in loops.items():
            closed[v].append(elapsed(lambda: window(ro)) / 80)

    # ---- evaluate() with K = 10, and the early exit, alternated
    def early_exit(ro, m=5):
        log = ro.eval_log
        log.begin()
        ro.reset()
        total, done = K * T, 0
        while done < total:
            n = min(16 * m, total - done)
            ro.run(n)
            done += n
            if int(log.count.min()) >= K:
                break
        return done

    wall = {(m, v): [] for m in ("greedy", "epsilon_greedy") for v in ("evaluate", "early_exit")}
    early_steps = {m: [] for m in ("greedy", "epsilon_greedy")}
    summaries, wasted = {}, {}
    for _ in range(args.rounds):
        for m in ("greedy", "epsilon_greedy"):
            ro = loops[(m, True)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ro.evaluate()
            torch.cuda.synchronize()
            wall[(m, "evaluate")].append((time.perf_counter() - t0) * 1e3)
            lengths = ro.eval_log.length.long().sum(1)
            wasted[m] = float((K * T - lengths).sum()) / (B * K * T)
            summaries[m] = ro.eval_log.summary()
            t0 = time.perf_counter()
            early_steps[m].append(early_exit(ro))
            torch.cuda.synchronize()
            wall[(m, "early_exit")].append((time.perf_counter() - t0) * 1e3)
    del loops

    # ---- the eval kernel alone: synthetic buffers, about 2 % of the envs finish per step
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
    env.reward.copy_(torch.rand_like(env.reward))
    env.dist.copy_(torch.rand_like(env.dist))
    env.done.copy_((torch.rand((B,), device="cuda:0") < 0.02).to(torch.uint8))
    log = EvalLog(env, K)

    def calls():
        log.begin()
        for _ in range(80):
            log.record()
    for _ in range(2):
        calls()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        calls()
    kernel_ms = [elapsed(g.replay, 5) / 81 for _ in range(args.rounds)]
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        calls()
        torch.cuda.synchronize()
    d = [e.device_time for e in prof.events() if "eval_kernel" in e.name]
    per_env = eval_bytes(0.02)

    # ---- bias of the windowed statistics: K = 1 against env.stats over the same T steps, greedy
    ev = make(cfg, sd, "greedy", False)
    ev_log = EvalLog(ev.env, 1)
    ev = Rollout(ev.env, ev.policy, use_graph=True, steps_per_graph=16, evaluate=ev_log)
    ev.evaluate()
    k1 = ev_log.summary()
    win = make(cfg, sd, "greedy", False)
    win.reset()
    win.env.stats.zero_()
    win.run(T)
    st = win.env.read_stats()

    med = {v: float(np.median(x)) for v, x in closed.items()}
    out = {
        "card": card(), "envs": B, "agents": B * N, "episodes_per_env": K, "max_episode_steps_plus_one": T,
        "rounds": args.rounds,
        "closed_loop_ms_per_env_step": {"%s/%s" % (m, "evaluate" if e else "plain"): stats(closed[(m, e)])
                                        for m, e in closed},
        "closed_loop_eval_overhead": {m: med[(m, True)] / med[(m, False)] - 1.0 for m in ("greedy", "epsilon_greedy")},
        "closed_loop_note": "PredatorCapturePrey_vdn checkpoint (hidden 128 GRU, tcgen05 kernel); epsilon-greedy: eps "
                            "0.05 flat; 16 env steps per graph; windows of 80 steps, each starting with mrb_eval_begin",
        "evaluate_k10_wall_ms": {"%s/%s" % k: stats(v) for k, v in wall.items()},
        "evaluate_note": "host clock around Rollout.evaluate() (begin, reset, %d env steps) and a synchronise; "
                         "early_exit: the same with count.min() read on the host every 80 steps" % (K * T),
        "early_exit_steps": {m: stats(v) for m, v in early_steps.items()},
        "steps_after_k_episodes_fraction": wasted,
        "steps_after_k_note": "env steps of evaluate() taken by envs that had already logged K episodes, over all "
                              "B * K * %d env steps" % T,
        "eval_call_us": float(np.median(kernel_ms)) * 1e3,
        "eval_call_note": "a graph of mrb_eval_begin + 80 mrb_eval_step calls over synthetic buffers (2 % of the envs "
                          "done), divided by 81 launches",
        "eval_kernel_us_profiler": {"median": float(np.median(d)) if d else None,
                                    "min": float(min(d)) if d else None, "max": float(max(d)) if d else None},
        "eval_bytes_per_env_step": per_env,
        "eval_hbm_floor_us": B * per_env / (HBM_TBPS * 1e12) * 1e6,
        "eval_floor_note": "bytes from shapes at 2 %% of envs finishing (reads reward, dist, done, accumulators; "
                           "writes accumulators; a finishing env also one row and its count) at %.1f TB/s" % HBM_TBPS,
        "summary_k10": summaries,
        "bias_k1_greedy": {"eval_return_mean": k1["return_mean"], "eval_episodes": k1["episodes"],
                           "windowed_stats_return_mean": st["return_sum"] / max(st["episodes"], 1.0),
                           "windowed_stats_episodes": st["episodes"],
                           "note": "K = 1: the first episode of every env; env.stats: every episode that finished in "
                                   "the first %d steps (auto-reset), same seed and policy" % T},
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
