"""ctypes binding of libmarbler_b200.so (include/marbler_b200.h).  There is no CPU fallback: if the
library cannot be loaded every entry point raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MARBLER_B200_LIB") or os.path.join(HERE, "libmarbler_b200.so")
ABI_VERSION = 7
NUM_STATS = 16
STAT_NAMES = ("episodes", "return_sum", "length_sum", "collisions", "boundary_exits", "scenario_metric",
              "env_steps", "qp_solves", "qp_iterations", "timeouts", "qp_stalls", "substeps", "qp_iterations_warp")
SYMBOLS = ("mrb_version", "mrb_create", "mrb_destroy", "mrb_last_error", "mrb_state_rows", "mrb_obs_dim",
           "mrb_num_actions", "mrb_bind", "mrb_reset", "mrb_step", "mrb_step_masked", "mrb_step_host", "mrb_barrier_qp",
           "mrb_get_state", "mrb_set_state", "mrb_fp64_peak", "mrb_launch_count", "mrb_policy_create", "mrb_policy_destroy", "mrb_policy_last_error", "mrb_policy_act",
           "mrb_policy_load", "mrb_select_actions", "mrb_record_begin", "mrb_record_step", "mrb_eval_begin",
           "mrb_eval_step")


class Spawn(C.Structure):
    _fields_ = [("count", C.c_int32), ("xr", C.c_int32), ("yr", C.c_int32), ("random_theta", C.c_int32),
                ("spacing", C.c_double), ("w2", C.c_double), ("h2", C.c_double),
                ("sx1", C.c_double), ("sx2", C.c_double), ("sy1", C.c_double), ("sy2", C.c_double)]


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "struct_size", "scenario", "num_robots", "update_frequency", "ctrl_period", "robotarium",
        "penalize_violations", "barrier_default", "max_episode_steps", "num_neighbors", "capability_aware",
        "num_prey", "num_predators", "n_fast", "small_torque", "large_torque", "auto_reset", "track_dist",
        "collect_stats", "reserved0")] + \
        [(n, C.c_double) for n in (
            "left", "right", "up", "down", "step_dist", "fast_step", "slow_step", "predator_radius",
            "capture_radius", "time_penalty", "sense_reward", "capture_reward", "load_reward", "unload_reward",
            "goal_width", "zone1_radius", "not_reached_penalty", "dist_multiplier", "reward_scaler",
            "violation_reward")] + \
        [("zone_mu", C.c_double * 2), ("zone_sigma", C.c_double * 2),
         ("spawn_robots", Spawn), ("spawn_other", Spawn),
         ("collision_diameter", C.c_double), ("collision_offset", C.c_double)]


class Buffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("state_f64", "state_i32", "obs", "reward", "done", "message",
                                          "remaining", "dist", "stats", "obs_f64", "reward_f64")]


# mrb_state_fields: (name, numpy dtype, shape per env as a function of (N, P)); order = the C struct
STATE_FIELDS = (
    ("poses", "f8", lambda N, P: (3, N)), ("prev_pose", "f8", lambda N, P: (3, N)), ("episode_return", "f8", lambda N, P: ()),
    ("episode_steps", "i4", lambda N, P: ()), ("prev_valid", "i4", lambda N, P: ()), ("episode_count", "i4", lambda N, P: ()),
    ("prey_loc", "f8", lambda N, P: (P, 2)), ("prey_sensed", "u1", lambda N, P: (P,)), ("prey_captured", "u1", lambda N, P: (P,)),
    ("loaded", "u1", lambda N, P: (N,)),
    ("load", "i4", lambda N, P: (N,)), ("zone_load", "i4", lambda N, P: (2,)), ("messages", "i4", lambda N, P: (4,)),
    ("grid", "u1", lambda N, P: (8, 12)), ("goal_col", "i4", lambda N, P: ()), ("pixel_type", "i4", lambda N, P: (N,)),
    ("reached_goal", "u1", lambda N, P: (N,)),
    ("goal", "f8", lambda N, P: (2,)),
)
COMMON_FIELDS = ("poses", "prev_pose", "episode_return", "episode_steps", "prev_valid", "episode_count")
SCENARIO_FIELDS = {"PredatorCapturePrey": ("prey_loc", "prey_sensed", "prey_captured"), "Warehouse": ("loaded",),
                   "MaterialTransport": ("load", "zone_load", "messages"),
                   "ArcticTransport": ("grid", "goal_col", "pixel_type", "reached_goal"), "Simple": ("goal",)}


class StateFields(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("reserved0", C.c_int32)] + [(n, C.c_void_p) for n, _, _ in STATE_FIELDS]


class PolicyDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("struct_size", "obs_dim", "input_dim", "hidden_dim", "n_actions", "n_agents",
                                         "obs_agent_id", "use_rnn", "non_shared", "accurate")]


SELECT_EPSILON_GREEDY, SELECT_SOFTMAX = 1, 2


class SelectDesc(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("mode", C.c_int32), ("seed", C.c_uint64), ("env_id0", C.c_int64),
                ("eps_start", C.c_double), ("eps_finish", C.c_double), ("anneal_time", C.c_int64)]


class EpisodeBatchDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("struct_size", "episode_limit", "obs_width", "reserved0")] + \
        [(n, C.c_void_p) for n in ("obs", "state", "actions", "actions_onehot", "avail_actions", "reward", "terminated",
                                   "filled", "cursor")]


class EvalTableDesc(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("episodes", C.c_int32)] + \
        [(n, C.c_void_p) for n in ("return_", "length", "message", "timeout", "remaining", "dist", "acc_return",
                                   "acc_length", "acc_dist", "count")]


_lib = None


def load():
    """Load the CUDA library (raises if it is missing: the product path has no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("marbler_b200: %s is missing - build it with `python -m marbler_b200.build` "
                           "(nvcc, sm_100a); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    sig = {
        "mrb_version": ([], C.c_int),
        "mrb_create": ([C.POINTER(Config), C.c_int, i64, i64, C.POINTER(vp)], C.c_int),
        "mrb_destroy": ([vp], C.c_int),
        "mrb_last_error": ([vp], C.c_char_p),
        "mrb_state_rows": ([vp, C.POINTER(i32), C.POINTER(i32)], C.c_int),
        "mrb_obs_dim": ([vp], C.c_int),
        "mrb_num_actions": ([vp], C.c_int),
        "mrb_bind": ([vp, C.POINTER(Buffers)], C.c_int),
        "mrb_reset": ([vp, vp, u64, vp], C.c_int),
        "mrb_step": ([vp, vp, vp], C.c_int),
        "mrb_step_masked": ([vp, vp, vp, vp], C.c_int),
        "mrb_step_host": ([vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "mrb_barrier_qp": ([C.c_int, i32, i32, i64, vp, vp, vp, vp, vp], C.c_int),
        "mrb_get_state": ([vp, i64, i64, C.POINTER(StateFields), vp], C.c_int),
        "mrb_set_state": ([vp, i64, i64, C.POINTER(StateFields), vp], C.c_int),
        "mrb_fp64_peak": ([C.c_int, C.c_double, C.POINTER(C.c_double)], C.c_int),
        "mrb_launch_count": ([], i64),
        "mrb_policy_create": ([C.POINTER(PolicyDesc), C.c_int, vp, i64, C.POINTER(vp)], C.c_int),
        "mrb_policy_destroy": ([vp], C.c_int),
        "mrb_policy_last_error": ([vp], C.c_char_p),
        "mrb_policy_act": ([vp, i64, vp, vp, vp, vp, vp, vp], C.c_int),
        "mrb_policy_load": ([vp, vp, i64, vp], C.c_int),
        "mrb_select_actions": ([C.c_int, i64, i32, i32, C.POINTER(SelectDesc), vp, vp, vp, vp], C.c_int),
        "mrb_record_begin": ([vp, C.POINTER(EpisodeBatchDesc), vp], C.c_int),
        "mrb_record_step": ([vp, C.POINTER(EpisodeBatchDesc), vp, vp], C.c_int),
        "mrb_eval_begin": ([vp, C.POINTER(EvalTableDesc), vp], C.c_int),
        "mrb_eval_step": ([vp, C.POINTER(EvalTableDesc), vp], C.c_int),
    }
    for name, (args, res) in sig.items():
        f = getattr(L, name)
        f.argtypes, f.restype = args, res
    if L.mrb_version() != ABI_VERSION:
        raise RuntimeError("marbler_b200: ABI version mismatch between _lib.py and %s" % LIB_PATH)
    _lib = L
    return L


def check_policy(rc, handle=None):
    if rc != 0:
        msg = load().mrb_policy_last_error(handle)
        raise RuntimeError("marbler_b200 policy error %d: %s" % (rc, (msg or b"").decode()))


def check(rc, handle=None):
    if rc != 0:
        msg = load().mrb_last_error(handle)
        raise RuntimeError("marbler_b200 error %d: %s" % (rc, (msg or b"").decode()))
