#!/usr/bin/env python
"""Headline benchmark: batched MARBLER env-steps/s on N B200s of one node (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scenario S] [--envs B]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one env step of every env of the batch (BASELINE.json configs[1]: PredatorCapturePrey-v0,
65,536 envs per GPU, barrier certificates on, random actions, auto-reset on done).  Envs are independent,
so N GPUs run N shards of B envs each with no data-path collective ("weak" scaling); the only
communication is the statistics all-reduce after the timed region.

Timing: CUDA events on the launch stream around every step; L2 is flushed (256 MiB memset) between
steps, outside the per-step events; `value` = world * B * K / max over ranks of the summed event time.
`e2e` = the same metric through the public host API (numpy actions in pinned memory -> H2D -> step ->
D2H obs/reward/done/message), wall clock with a synchronize on both sides.
`--impl reference` times the CPU path: the C restatement of the reference (oracle/, kind "port" - the
reference itself is Python that needs rps/cvxopt/gym, none of which exist on the GPU box) on all host
threads.  The oracle is only ever the checker / the CPU baseline here, never the product path.
`--dump-outputs DIR` writes what the last timed step returned to its caller (obs, reward, done, message; rank 0's
shard) as DIR/<name>.npy in float32, so that two builds run with the same arguments can be compared output for
output: reset seeds and actions are fixed, so the inputs are the same from run to run.  DIR/env_index.npy names the
env of every row; above 64 MB in all, a fixed, seeded sample of envs is written instead of every env.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FALLBACK_HBM_GBS = 6650.0            # /opt/skills/guides/B200_PROFILING.md fallback
METRIC = "batched env-steps/s (PredatorCapturePrey-v0, barrier certs on)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenario", default="PredatorCapturePrey")
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--override", action="append", default=[], help="config key=value (python literal)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not bind the process to the CPUs next to its GPU")
    ap.add_argument("--rollout", action="store_true",
                    help="also time the closed loop policy kernel -> step kernel (SURVEY 8f-1), random-init GRU agent")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times a host-dependent sample of envs)")
    return args


def load_cfg(args):
    from marbler_b200 import config
    cfg = config.load_yaml(config.default_config_path(args.scenario))
    for kv in args.override:
        k, v = kv.split("=", 1)
        cfg[k] = eval(v)
    return cfg


def workload_name(args, cfg, world):
    return "%s-v0 batched %d envs/GPU x %d GPU, random actions, barrier_certificate=%s, auto-reset" % (
        args.scenario, args.envs, world, cfg.get("barrier_certificate", "safe"))


def layout_bytes_per_env_step(env):
    """HBM bytes one env step moves with THIS layout (DESIGN.md section 4): state rows read and written once, actions
    in, obs / reward / done / message / remaining / dist out - SURVEY 8(d)'s figure plus the rows it calls optional
    (previous pose, dist_travelled, episode return, episode counter)."""
    N, D = env.N, env.D
    rf, ri = env.state_f64.shape[0], env.state_i32.shape[0]
    read = 8 * rf + 4 * ri + 4 * N
    write = 8 * (5 * N + 1) + 4 * ri + 4 * N * D + 4 * N + 1 + 1 + 4 + (4 * N if env.dist is not None else 0)
    return read + write


def algorithmic_bytes_per_env_step(scenario, N, D, P):
    """SURVEY.md 8(d): 48N (pose r+w) + 4N (actions) + 4*N*D (obs) + rewards + 2 (done, message) + scenario state.
    PCP 582, Warehouse 782, MaterialTransport 422, ArcticTransport 818, Simple 410, PCP-20 2,438 B."""
    base = 48 * N + 4 * N + 4 * N * D + 2
    return base + {"PredatorCapturePrey": 4 + 16 * P + 16, "Warehouse": 4 * N + 12, "MaterialTransport": 4 + 64,
                   "ArcticTransport": 4 + 96 + 28, "Simple": 4 * N + 16 + 8}[scenario]


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._halt.set()
        self.join(2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def cpu_port_rate(args, cfg, seconds, envs=None):
    """env-steps/s of the C restatement of the reference on all host threads (bounded sample)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import c_oracle
    cores = os.cpu_count() or 1
    orc = c_oracle.COracle(args.scenario, cfg)
    B = envs or max(cores * 1024, 16384)
    sf, si = orc.reset_flat(B, seed=0, threads=cores)
    rng = np.random.RandomState(0)
    acts = [rng.randint(0, orc.n_actions, size=(B, orc.N)).astype(np.int32) for _ in range(8)]
    for i in range(2):
        orc.step_flat(sf, si, acts[i], auto_reset=True, threads=cores)
    t0, n = time.perf_counter(), 0
    while True:
        orc.step_flat(sf, si, acts[n % 8], auto_reset=True, threads=cores)
        n += 1
        dt = time.perf_counter() - t0
        if dt > seconds or n >= 10000:
            break
    return {"value": B * n / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": "%d envs x %d steps of the same workload (%.1f s), C restatement of the reference "
                      "(oracle/marbler_oracle.c), %d host threads" % (B, n, dt, cores)}, B, n, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = load_cfg(args)
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    # bounded sample per step: at most ~0.2 s of CPU work per step, never more than the workload
    probe, _, _, _ = cpu_port_rate(args, cfg, 1.0)
    sample = int(min(args.envs, max(1024, probe["value"] * 0.2)))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import c_oracle
    cores = os.cpu_count() or 1
    orc = c_oracle.COracle(args.scenario, cfg)
    sf, si = orc.reset_flat(sample, seed=0, threads=cores)
    rng = np.random.RandomState(0)
    acts = [rng.randint(0, orc.n_actions, size=(sample, orc.N)).astype(np.int32) for _ in range(args.warmup + args.steps)]
    for i in range(args.warmup):
        orc.step_flat(sf, si, acts[i], auto_reset=True, threads=cores)
    t0 = time.perf_counter()
    for i in range(args.steps):
        orc.step_flat(sf, si, acts[args.warmup + i], auto_reset=True, threads=cores)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    desc = "%d envs per step (bounded sample of the %d-env workload), %d steps, C restatement of the reference " \
           "(oracle/marbler_oracle.c; the Python reference needs rps/cvxopt/gym which are not installable), " \
           "%d host threads" % (sample, args.envs, args.steps, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC if args.scenario == "PredatorCapturePrey" else "batched env-steps/s (%s)" % args.scenario,
        "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": {"workload": workload_name(args, cfg, world)},
        "agent_steps_per_s": value * orc.N,
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def time_rollout(env, steps):
    """Closed loop on the device: policy kernel (fc1 -> GRUCell -> fc2 -> argmax, the reference's RNNAgent with
    hidden_dim 128 and obs_agent_id, random-init weights) -> step kernel, replayed from a CUDA graph."""
    import torch
    from marbler_b200.policy import Policy, Rollout
    g = torch.Generator().manual_seed(0)
    H, Din, A = 128, env.D + env.N, env.n_actions
    u = lambda *shape: (torch.rand(shape, generator=g) * 2 - 1) / (shape[-1] ** 0.5)
    sd = {"fc1.weight": u(H, Din), "fc1.bias": u(H), "rnn.weight_ih": u(3 * H, H), "rnn.weight_hh": u(3 * H, H),
          "rnn.bias_ih": u(3 * H), "rnn.bias_hh": u(3 * H), "fc2.weight": u(A, H), "fc2.bias": u(A)}
    pol = Policy(sd, env.N, env.D, obs_agent_id=True, device=env.device)
    ro = Rollout(env, pol, use_graph=True, steps_per_graph=16)
    ro.reset()
    ro.run(33)
    steps = max(16, steps // 16 * 16)
    e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    torch.cuda.synchronize()
    e0.record()
    ro.run(steps)
    e1.record()
    for _ in range(20):
        pol.act(env.obs, ro.hidden, actions=ro.actions, fresh=env.done)
    e2.record()
    for _ in range(20):
        env.step(ro.actions)
    e3.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    flops = 2.0 * env.B * env.N * (H * Din + 6 * H * H + H * A)
    pol_ms = e1.elapsed_time(e2) / 20
    return {"env_steps_per_s": env.B / (ms * 1e-3), "ms_per_step": ms, "policy_kernel_ms": pol_ms,
            "step_kernel_ms": e2.elapsed_time(e3) / 20, "policy_tflops": flops / (pol_ms * 1e-3) / 1e12,
            "steps": steps, "kernels_per_step": 2, "launch": "CUDA graph replay, 16 env steps per graph",
            "policy": "RNNAgent hidden 128, GRUCell, obs_agent_id, greedy; persistent tcgen05 / TMEM kernel, FP16 operands, FP32 accumulate; random-init weights"}


def pcie_floor(env, world, barrier, reps=10):
    """Bare pinned device->host copy of one step's outputs, all ranks at once: the floor of the e2e path."""
    import torch
    n = env.d2h_bytes_per_step
    src = torch.empty(n, dtype=torch.uint8, device=env.device)
    dst = torch.empty(n, dtype=torch.uint8).pin_memory()
    for _ in range(2):
        dst.copy_(src, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=env.device)
    if world > 1:
        torch.distributed.all_reduce(dt, op=torch.distributed.ReduceOp.MAX)
    per = float(dt.item()) / reps
    return {"d2h_ms_per_step": per * 1e3, "aggregate_gbs": world * n / per / 1e9, "bytes_per_gpu": n,
            "env_steps_per_s_at_floor": world * env.B / per,
            "how": "every rank copies one step's outputs (obs + reward + done + message) device -> pinned host, "
                   "%d times back to back, all ranks at once; max over ranks" % reps}


DUMP_LIMIT_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, outputs):
    """outputs: name -> CUDA tensor with a leading env axis.  Writes each as out_dir/<name>.npy in float32 (done and
    message are small integers, exact there) plus env_index.npy, the env of every row.  When everything would exceed
    DUMP_LIMIT_BYTES, every array keeps the same fixed, seeded sample of envs."""
    import numpy as np
    B = next(iter(outputs.values())).shape[0]
    per_env = 8 + sum(4 * t[0].numel() for t in outputs.values())      # 8: the float64 env index
    budget = DUMP_LIMIT_BYTES - 4096                                      # .npy headers
    index = np.arange(B)
    if B * per_env > budget:
        index = np.sort(np.random.RandomState(0).choice(B, budget // per_env, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy()[index].astype(np.float32))
    np.save(os.path.join(out_dir, "env_index.npy"), index.astype(np.float64))


def run_ours(args):
    import numpy as np
    import torch
    from marbler_b200 import build, sharding
    from marbler_b200.vec_env import VecEnv
    from marbler_b200 import flop_model
    from marbler_b200.vec_env import fp64_peak
    build.build()
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
    # run on the CPUs next to this rank's GPU BEFORE anything allocates pinned memory (first touch decides the NUMA
    # node of the host buffers the e2e path copies into); the full mask is restored for the CPU baseline leg
    all_cpus = os.sched_getaffinity(0)
    numa = sharding.bind_to_gpu_numa(int(os.environ.get("LOCAL_RANK", "0"))) if not args.no_numa_bind else None
    rank, world, local = sharding.init_distributed()
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    fp64_tflops = fp64_peak(local, 150.0)       # measured DFMA rate of this GPU: the denominator of the binding roofline
    cfg = load_cfg(args)
    B, K, W = args.envs, args.steps, args.warmup
    env = VecEnv(args.scenario, cfg, num_envs=B, device=dev, seed=0, env_id0=rank * B, auto_reset=True)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    n_pool = min(W + K, 64)
    acts = [torch.randint(0, env.n_actions, (B, env.N), generator=gen, device=dev, dtype=torch.int32) for _ in range(n_pool)]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for i in range(W):
        env.step(acts[i % n_pool])
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    sampler = ClockSampler(local)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    env.stats.zero_()
    barrier()
    launches0 = env.lib.mrb_launch_count()
    sampler.start()
    wall0 = time.perf_counter()
    for i in range(K):
        flush.zero_()                                   # L2 flush, outside the per-step events
        starts[i].record()
        env.step(acts[(W + i) % n_pool])
        ends[i].record()
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    launches = env.lib.mrb_launch_count() - launches0
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    stats = sharding.summarize(sharding.allreduce_stats(env.stats))
    if args.dump_outputs and rank == 0:                 # before the e2e leg below steps the env again
        dump_outputs(args.dump_outputs, {"obs": env.obs, "reward": env.reward, "done": env.done, "message": env.message})

    # ---- end to end through the host API: pinned numpy actions -> H2D -> step -> D2H -> sync
    Ke = max(3, min(K, 50))
    h = env.host_buffers()
    rng = np.random.RandomState(rank)
    # four pinned action batches, written before the clock starts (a host-side policy writes its actions into pinned
    # memory itself); every timed step uploads one of them, runs the step and brings obs/reward/done/message back
    host_actions = [torch.from_numpy(rng.randint(0, env.n_actions, size=(B, env.N)).astype(np.int32)).pin_memory()
                    for _ in range(4)]
    for i in range(3):
        env.step_host(host_actions[i % 4])
    barrier()
    t0 = time.perf_counter()
    for i in range(Ke):
        env.step_host(host_actions[i % 4])
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(e2e_s, op=torch.distributed.ReduceOp.MAX)
    e2e_rate = world * B * Ke / float(e2e_s.item())
    floor = pcie_floor(env, world, barrier)

    rollout = time_rollout(env, min(K, 320)) if args.rollout else None
    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    value = world * B * K / (dev_ms_max * 1e-3)
    ms_per_step = dev_ms_max / K
    bytes_step = algorithmic_bytes_per_env_step(args.scenario, env.N, env.D, env.P)
    flops = flop_model.flops(args.scenario, env.N, stats)          # stats: summed over ranks, timed region only
    fp64_achieved = None if flops is None else flops["total"] / world / (dev_ms_max * 1e-3) / 1e12      # per GPU
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_kind = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md, 6.65 TB/s)"
    if os.path.exists(peaks_path):
        try:
            peak = float(json.load(open(peaks_path))["hbm_gbs"])
            peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    achieved = bytes_step * B / (ms_per_step * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("%s_%d" % (args.scenario, B))
        except Exception:
            pass
    out = {
        "metric": METRIC if args.scenario == "PredatorCapturePrey" else "batched env-steps/s (%s)" % args.scenario,
        "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, cfg, world), "envs_per_gpu": B, "robots_per_env": env.N,
                   "l2": "flushed between steps (256 MiB memset outside the per-step CUDA events)",
                   "timing": "sum of per-step CUDA event durations, max over ranks",
                   "wall_s_timed_region_incl_flush": wall},
        "agent_steps_per_s": value * env.N,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_kind": peak_kind, "bytes_per_env_step": bytes_step,
                     "bytes_layout": layout_bytes_per_env_step(env),
                     "kernel": "%s<%s,%d>" % ("step_thread_kernel" if env.N <= 6 else "step_warp_kernel", args.scenario, env.N),
                     "note": "bytes_per_env_step is SURVEY 8(d)'s figure; bytes_layout adds the optional rows this layout "
                             "keeps.  The step is FP64-issue bound, not HBM bound (SURVEY 8d): roofline_fp64 is the "
                             "binding roofline"},
        "roofline_fp64": None if flops is None else {
            "bound": "fp64", "achieved": fp64_achieved, "peak": fp64_tflops, "unit": "TFLOP/s",
            "frac": fp64_achieved / fp64_tflops,
            "flops_per_env_step": flops["total"] / max(stats["env_steps"], 1.0),
            "peak_kind": "measured in this run: mrb_fp64_peak (independent DFMA chains, best launch)",
            "model": flops["model"], "per_gpu": True},
        "fp64": {"ipm_iterations_per_solve": stats["qp_iters_per_solve"],
                 "qp_solves_per_env_step": stats["qp_solves"] / max(stats["env_steps"], 1.0),
                 "substeps_per_env_step": stats["substeps"] / max(stats["env_steps"], 1.0),
                 "qp_stalls": stats["qp_stalls"],
                 # iterations the warps ran / iterations the envs needed (one env per thread: a warp waits for its
                 # slowest env): the divergence overhead of the solver loop
                 "warp_iteration_overhead": stats["qp_iterations_warp"] / max(stats["qp_iterations"], 1.0)},
        "episodes": {k: stats[k] for k in ("episodes", "return_mean", "length_mean", "collisions", "boundary_exits", "timeouts")},
        "clocks": clocks,
        "e2e": {"value": e2e_rate, "unit": "env-steps/s", "h2d_bytes_per_step": env.h2d_bytes_per_step * world,
                "d2h_bytes_per_step": env.d2h_bytes_per_step * world, "steps": Ke,
                "api": "VecEnv.step_host -> mrb_step_host (pinned host buffers, one sync per step)",
                "pcie_floor": floor, "cpu_affinity": numa},
        "gpu_launches": int(launches),
    }
    if args.rollout:
        out["rollout"] = rollout
    if world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)       # the CPU leg gets every host core back
        out["cpu_baseline"], _, _, _ = cpu_port_rate(args, cfg, args.cpu_seconds)
    print(json.dumps(out))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
