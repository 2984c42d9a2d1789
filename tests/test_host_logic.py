"""CPU-only tests of the host layer: the C-ABI library loads and exports every symbol the header
declares (no compute without a GPU), config derivation, state packing, registry / spaces, sharding."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import golden_util as gu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from marbler_b200 import build, _lib
    build.build()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from marbler_b200 import _lib
    header = open(os.path.join(ROOT, "include", "marbler_b200.h")).read()
    declared = set(re.findall(r"\b(mrb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS)
    raw = C.CDLL(_lib.LIB_PATH)
    for s in declared:
        assert hasattr(raw, s), s
    assert lib.mrb_version() == _lib.ABI_VERSION


def test_create_fails_loudly_without_gpu(lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from marbler_b200 import _lib, config
    c = config.make_config("PredatorCapturePrey", config.load_yaml(config.default_config_path("PredatorCapturePrey")))
    h = C.c_void_p()
    rc = lib.mrb_create(C.byref(c), 0, 16, 0, C.byref(h))
    assert rc == -2 and b"no CUDA device" in lib.mrb_last_error(None)
    with pytest.raises(RuntimeError):
        import marbler_b200
        marbler_b200.make("PredatorCapturePrey-v0")


def test_create_rejects_bad_configs(lib):
    from marbler_b200 import config
    cfg = config.load_yaml(config.default_config_path("PredatorCapturePrey"))
    c = config.make_config("PredatorCapturePrey", cfg)
    c.struct_size = 8
    h = C.c_void_p()
    assert lib.mrb_create(C.byref(c), 0, 16, 0, C.byref(h)) == -1
    assert b"ABI" in lib.mrb_last_error(None)
    # a single robot has no pair constraint (and the warp kernel's pair decode assumes N >= 2)
    one = config.make_config("Simple", dict(config.load_yaml(config.default_config_path("Simple")), n_agents=1))
    assert lib.mrb_create(C.byref(one), 0, 16, 0, C.byref(h)) == -1 and b"[2, 32]" in lib.mrb_last_error(None)
    bad = config.make_config("PredatorCapturePrey", dict(cfg, rps_collision_diameter=0.0))
    assert lib.mrb_create(C.byref(bad), 0, 16, 0, C.byref(h)) == -1 and b"collision_diameter" in lib.mrb_last_error(None)
    with pytest.raises(ValueError):                     # rps asserts the spawn grid has room (SURVEY a14)
        config.make_config("PredatorCapturePrey", dict(cfg, predator=10, capture=10))
    with pytest.raises(ValueError):
        config.make_config("PredatorCapturePrey", dict(cfg, barrier_certificate="custom"))


@pytest.mark.parametrize("name", gu.fixture_names())
def test_config_matches_oracle_config(oracle_lib, name):
    """Product and oracle derive their configs independently from the same YAML dict."""
    from marbler_b200 import config
    g = gu.Golden(name)
    mine = config.make_config(g.scenario, g.cfg)
    ref = oracle_lib.make_config(g.scenario, g.cfg)
    pairs = [("num_robots", "N"), ("left", "LEFT"), ("right", "RIGHT"), ("up", "UP"), ("down", "DOWN")]
    for a, b in pairs:
        assert getattr(mine, a) == getattr(ref, b)
    same = ["scenario", "update_frequency", "ctrl_period", "robotarium", "penalize_violations", "barrier_default",
            "max_episode_steps", "num_neighbors", "capability_aware", "num_prey", "num_predators", "n_fast",
            "small_torque", "large_torque", "step_dist", "fast_step", "slow_step", "predator_radius",
            "capture_radius", "time_penalty", "sense_reward", "capture_reward", "load_reward", "unload_reward",
            "goal_width", "zone1_radius", "not_reached_penalty", "dist_multiplier", "reward_scaler", "violation_reward",
            "collision_diameter", "collision_offset"]
    for k in same:
        assert getattr(mine, k) == getattr(ref, k), k
    for sp in ("spawn_robots", "spawn_other"):
        for f, _ in mine.spawn_robots._fields_:
            assert getattr(getattr(mine, sp), f) == getattr(getattr(ref, sp), f), (sp, f)


@pytest.mark.parametrize("name", gu.fixture_names())
def test_state_pack_roundtrip(name):
    from marbler_b200 import layout
    g = gu.Golden(name)
    N = g.s0["poses"].shape[2]
    P = g.s0["prey_loc"].shape[1] if "prey_loc" in g.s0 else 0
    sf, si = layout.pack(g.scenario, N, P, g.s0, g.B)
    assert sf.shape[0], si.shape[0] == layout.rows(g.scenario, N, P)
    back = layout.unpack(g.scenario, N, P, sf, si)
    for k, v in g.s0.items():
        if k == "prev_pose":
            assert np.array_equal(back[k][:, :2], v[:, :2])
        else:
            assert np.array_equal(np.asarray(back[k]).astype(np.float64), np.asarray(v).astype(np.float64)), k


def test_registry_keys_and_space_dims():
    """Same five gym ids as robotarium_gym/__init__.py:4-10; obs / action dims equal the dimensions
    the reference's shipped checkpoints pin (SURVEY.md section 4 table)."""
    import marbler_b200
    from marbler_b200 import config
    assert set(marbler_b200.registry) == {"PredatorCapturePrey-v0", "Warehouse-v0", "Simple-v0",
                                          "ArcticTransport-v0", "MaterialTransport-v0"}
    want = {"PredatorCapturePrey": (16, 4), "Warehouse": (18, 6), "MaterialTransport": (9, 4),
            "ArcticTransport": (30, 4), "Simple": (10, 4)}
    for scn, (d, n) in want.items():
        cfg = config.load_yaml(config.default_config_path(scn))
        c = config.make_config(scn, cfg)
        assert (config.obs_space_dim(scn, cfg, c), c.num_robots) == (d, n)


def test_default_configs_equal_reference_yaml():
    """Against the config each scenario's rollout fixture was made with: the reference's own config.yaml with the
    overrides of oracle/ref_harness.py reference_config() (figures, gif, logging, real time and robotarium off) and a
    seed of the fixture's own (oracle/gen_golden.py), so the seed is not compared."""
    from marbler_b200 import config
    for scn in config.SCENARIOS:
        ref = gu.Golden(scn + "_rollout").cfg
        mine = config.load_yaml(config.default_config_path(scn))
        for k, v in mine.items():
            if k in ("show_figure_frequency", "save_gif", "real_time", "seed"):
                continue
            assert ref[k] == v, (scn, k)


def test_shard_range_partitions():
    from marbler_b200.sharding import shard_range
    for total in (1, 7, 65536, 1048576, 1000003):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == total
            for (s0, c0), (s1, _) in zip(spans, spans[1:]):
                assert s0 + c0 == s1
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1


def _worker(rank, world, port, q):
    import torch.distributed as dist
    from marbler_b200.sharding import allreduce_stats, shard_range, summarize
    from marbler_b200._lib import NUM_STATS
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    start, count = shard_range(1001, rank, world)
    st = torch.zeros(NUM_STATS, dtype=torch.float64)
    st[0], st[1], st[2], st[6] = count, 2.0 * count, 10.0 * count, start
    red = allreduce_stats(st)
    q.put((rank, red.tolist(), summarize(red)))
    dist.destroy_process_group()


def test_stats_allreduce_two_ranks_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=120) for _ in procs)
    [p.join(60) for p in procs]
    for rank, vec, summ in res:
        assert vec[0] == 1001 and vec[1] == 2002 and vec[6] == 501
        assert summ["return_mean"] == 2.0 and summ["length_mean"] == 10.0


def test_spawn_grid_division_trick_is_exact():
    """csrc/step_thread.cuh spawn_grid: cell // yr as (cell * ceil(65536 / yr)) >> 16 for every grid the library accepts
    (at most 64 cells)."""
    for yr in range(1, 65):
        inv = (65536 + yr - 1) // yr
        for cell in range(64):
            assert (cell * inv) >> 16 == cell // yr, (cell, yr)


def test_team_kernel_table_matches_the_units():
    """csrc/launchers.h states which (scenario, size of the Newton system) has a kernel with the FP64 tensor-core solver:
    n = 8, 12, ..., team_kernel_max(scenario).  The units kern_team_<scenario><n>.cu must be exactly those, each must
    instantiate the step launcher of its size, and each PredatorCapturePrey unit also the QP-alone launcher mrb_barrier_qp
    uses."""
    import glob
    import re
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "marbler_b200", "csrc")
    table = re.search(r"constexpr int team_kernel_max\(int scn\) \{ return (.*?); \}", open(os.path.join(csrc, "launchers.h")).read()).group(1)
    tags = {"MRB_PCP": "pcp", "MRB_WAREHOUSE": "warehouse", "MRB_SIMPLE": "simple"}
    maxima = {scn: int(n) for scn, n in re.findall(r"scn == (\w+) \? (\d+)", table)}
    assert table.endswith(": 0") and set(maxima) == set(tags) and all(8 <= top <= 32 for top in maxima.values()), table
    want = {(scn, n) for scn, top in maxima.items() for n in range(8, top + 1, 4)}
    units = {os.path.basename(u): u for u in glob.glob(os.path.join(csrc, "kern_team_*.cu"))}
    assert set(units) == {"kern_team_%s%d.cu" % (tags[scn], n) for scn, n in want}, sorted(units)
    for scn, n in want:
        src = open(units["kern_team_%s%d.cu" % (tags[scn], n)]).read()
        assert "template cudaError_t launch_step_team<%s, %d>(" % (scn, n) in src, (scn, n)
        assert ("template cudaError_t launch_qp_team<%d>(" % n in src) == (scn == "MRB_PCP"), (scn, n)
