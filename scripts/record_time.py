"""Cost of episode recording (mrb_record_begin / mrb_record_step), measured in one process with the variants alternated:

  * the epsilon-greedy closed loop (policy -> selection -> step [-> record], CUDA-graph replays of 16 env steps) on
    65,536 PredatorCapturePrey envs with the shipped hidden-128 GRU checkpoint, with and without recording, as time
    per env step (each timed window of 80 steps starts with mrb_record_begin, so every recorded step writes an active
    row);
  * a whole 81-step collect() (begin, reset, 81 env steps) against the same loop without recording;
  * the record kernel alone (a graph of begin + 81 record calls over synthetic data in which no env finishes, so
    every call writes every field), against its HBM floor from the bytes the shapes imply, and the kernel's own
    duration from a profiler pass;
  * the alternative design, zero-filling the whole batch at mrb_record_begin, as the time of that fill.

Usage: python scripts/record_time.py [--out FILE.json]   (prints the JSON either way; needs a B200)."""
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
from marbler_b200.policy import EpisodeBatch, Exploration, Policy, Rollout  # noqa: E402
from marbler_b200.vec_env import VecEnv  # noqa: E402

B, N, D, A, T = 65536, 4, 16, 5, 81
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


def record_bytes(W):
    """Bytes one mrb_record_step moves per env when the env is active: reads obs, reward, done, actions, cursor;
    writes obs row (W wide), actions (int64), one-hot, avail_actions, reward, terminated, filled, cursor."""
    read = 4 * N * D + 4 * N + 1 + 4 * N + 4
    write = 4 * N * W + 8 * N + 4 * N * A + 4 * N * A + 4 + 1 + 8 + 4
    return read + write


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    cfg = dict(gu.Golden("PredatorCapturePrey_rollout").cfg)
    z = np.load(os.path.join(gu.GOLDEN, "policy", "PredatorCapturePrey_vdn.npz"))
    sd = {k[3:]: z[k] for k in z.files if k.startswith("sd.")}

    # ---- closed loop, with and without recording
    loops = {}
    for v in ("plain", "record"):
        env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
        ex = Exploration("epsilon_greedy", seed=1, eps_start=0.05, eps_finish=0.05, device="cuda:0")
        rec = EpisodeBatch(env, T) if v == "record" else None
        ro = Rollout(env, Policy(sd, N, D, device="cuda:0"), use_graph=True, steps_per_graph=16, explore=ex, record=rec)
        ro.collect() if rec is not None else (ro.reset(), ro.run(T))
        loops[v] = ro
    torch.cuda.synchronize()

    def window(ro):
        if ro.record is not None:
            ro.record.begin()
        for _ in range(5):
            ro.run(16)

    closed = {v: [] for v in loops}
    collect = {v: [] for v in loops}
    for _ in range(args.rounds):
        for v, ro in loops.items():
            closed[v].append(elapsed(lambda: window(ro)) / 80)
        for v, ro in loops.items():
            collect[v].append(elapsed(ro.collect if ro.record is not None else (lambda: (ro.reset(), ro.run(T)))))
    W = loops["record"].record.obs_width
    del loops

    # ---- the record kernel alone: synthetic buffers in which no env finishes
    env = VecEnv("PredatorCapturePrey", cfg, num_envs=B, device="cuda:0", seed=3, auto_reset=True)
    env.obs.copy_(torch.rand_like(env.obs))
    env.reward.copy_(torch.rand_like(env.reward))
    env.done.zero_()
    actions = torch.randint(0, A, (B, N), dtype=torch.int32, device="cuda:0")
    rec = EpisodeBatch(env, T)

    def calls():
        rec.begin()
        for _ in range(T):
            rec.record(actions)
    for _ in range(2):
        calls()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        calls()
    kernel_ms = []
    fill_ms = []
    tensors = [t for k, t in rec.data.items() if k != "state"]
    fill = lambda: [t.zero_() for t in tensors]
    fill()
    for _ in range(args.rounds):
        kernel_ms.append(elapsed(g.replay, 5) / (T + 1))
        fill_ms.append(elapsed(fill, 5))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        calls()
        torch.cuda.synchronize()
    d = [e.device_time for e in prof.events() if "record_kernel" in e.name]
    per_env = record_bytes(W)
    batch_bytes = sum(t.numel() * t.element_size() for t in tensors)

    med = {v: float(np.median(x)) for v, x in closed.items()}
    cmed = {v: float(np.median(x)) for v, x in collect.items()}
    kmed = float(np.median(kernel_ms))
    out = {
        "card": card(), "envs": B, "agents": B * N, "episode_limit": T, "obs_width": W, "rounds": args.rounds,
        "closed_loop_ms_per_env_step": {v: {"median": med[v], "min": float(min(closed[v])), "max": float(max(closed[v]))}
                                        for v in med},
        "closed_loop_record_overhead": med["record"] / med["plain"] - 1.0,
        "closed_loop_note": "PredatorCapturePrey_vdn checkpoint (hidden 128 GRU, tcgen05 kernel); epsilon-greedy, eps "
                            "0.05 flat; 16 env steps per graph; windows of 80 steps, each starting with mrb_record_begin",
        "collect_81_steps_ms": {v: {"median": cmed[v], "min": float(min(collect[v])), "max": float(max(collect[v]))}
                                for v in cmed},
        "collect_note": "record: Rollout.collect() (begin, reset, 81 steps); plain: reset + run(81) without recording",
        "record_call_us": kmed * 1e3,
        "record_call_note": "a graph of mrb_record_begin + 81 mrb_record_step calls over synthetic buffers in which "
                            "no env finishes, divided by 82 launches",
        "record_kernel_us_profiler": {"median": float(np.median(d)) if d else None,
                                      "min": float(min(d)) if d else None, "max": float(max(d)) if d else None},
        "record_bytes_per_env_step": per_env,
        "record_hbm_floor_us": B * per_env / (HBM_TBPS * 1e12) * 1e6,
        "record_floor_note": "bytes from shapes (reads obs, reward, done, actions, cursor; writes the row of every "
                            "field and the cursor) at %.1f TB/s" % HBM_TBPS,
        "zero_fill_alternative": {"batch_bytes": batch_bytes, "fill_ms_per_collection": float(np.median(fill_ms)),
                                  "fill_us_per_env_step": float(np.median(fill_ms)) * 1e3 / T,
                                  "note": "torch zero_() of every batch tensor: what zeroing the batch at "
                                          "mrb_record_begin would add to each collection"},
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
