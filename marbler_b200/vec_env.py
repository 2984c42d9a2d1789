"""Batched environment core: owns the PyTorch device buffers and one libmarbler_b200 handle.

This is the thin host layer between the reference-facing classes (wrapper.py, scenarios/) and the
C ABI.  PyTorch provides device memory and streams only; every number is produced by the CUDA kernels
behind mrb_step / mrb_reset.  There is no CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, layout
from .config import SCENARIOS, make_config


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class VecEnv(object):
    def __init__(self, scenario, cfg, num_envs=1, device=None, seed=0, env_id0=0, auto_reset=False,
                 track_dist=True, collect_stats=True, f64_outputs=False):
        if not torch.cuda.is_available():
            raise RuntimeError("marbler_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.scenario = scenario
        self.cfg = dict(cfg)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("marbler_b200: device must be a CUDA device")
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)
        self.c = make_config(scenario, cfg, auto_reset=auto_reset, track_dist=track_dist, collect_stats=collect_stats)
        self.B, self.N, self.P = int(num_envs), int(self.c.num_robots), int(self.c.num_prey)
        self.seed = int(seed) & (2 ** 64 - 1)
        self.env_id0 = int(env_id0)
        self.handle = C.c_void_p()
        _lib.check(self.lib.mrb_create(C.byref(self.c), dev_index, self.B, self.env_id0, C.byref(self.handle)))
        rf, ri = C.c_int32(), C.c_int32()
        _lib.check(self.lib.mrb_state_rows(self.handle, C.byref(rf), C.byref(ri)), self.handle)
        assert (rf.value, ri.value) == layout.rows(scenario, self.N, self.P)
        self.D = self.lib.mrb_obs_dim(self.handle)
        self.n_actions = self.lib.mrb_num_actions(self.handle)
        B, N, D, dev = self.B, self.N, self.D, self.device
        self.state_f64 = torch.zeros((rf.value, B), dtype=torch.float64, device=dev)
        self.state_i32 = torch.zeros((ri.value, B), dtype=torch.int32, device=dev)
        self.obs = torch.zeros((B, N, D), dtype=torch.float32, device=dev)
        self.reward = torch.zeros((B, N), dtype=torch.float32, device=dev)
        self.done = torch.zeros((B,), dtype=torch.uint8, device=dev)
        self.message = torch.zeros((B,), dtype=torch.uint8, device=dev)
        self.remaining = torch.zeros((B,), dtype=torch.int32, device=dev)
        self.dist = torch.zeros((B, N), dtype=torch.float32, device=dev) if track_dist else None
        self.stats = torch.zeros((_lib.NUM_STATS,), dtype=torch.float64, device=dev)
        # float64 copies of obs / reward (the reference's own precision; used by the single-env drop-in path)
        self.obs_f64 = torch.zeros((B, N, D), dtype=torch.float64, device=dev) if f64_outputs else None
        self.reward_f64 = torch.zeros((B, N), dtype=torch.float64, device=dev) if f64_outputs else None
        self._buffers = _lib.Buffers(*[_ptr(t).value for t in (
            self.state_f64, self.state_i32, self.obs, self.reward, self.done, self.message, self.remaining,
            self.dist, self.stats, self.obs_f64, self.reward_f64)])
        _lib.check(self.lib.mrb_bind(self.handle, C.byref(self._buffers)), self.handle)
        self._host = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.mrb_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ reset / step
    def reset(self, mask=None, seed=None):
        """Re-sample the masked envs (all when mask is None).  Returns the (zeroed) obs buffer."""
        if seed is not None:
            self.seed = int(seed) & (2 ** 64 - 1)
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            assert m.shape == (self.B,)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrb_reset(self.handle, _ptr(m), self.seed, self._stream()), self.handle)
        return self.obs

    def active_mask(self, active):
        """The u8 [B] view mrb_step_masked reads of `active`, a bool or uint8 tensor [B] on the env's device (no copy
        when it is contiguous).  TypeError / ValueError otherwise, before any device work."""
        if not isinstance(active, torch.Tensor) or active.dtype not in (torch.bool, torch.uint8):
            raise TypeError("active must be a bool or uint8 tensor, not %r" % (getattr(active, "dtype", type(active)),))
        if tuple(active.shape) != (self.B,):
            raise ValueError("active must have shape (%d,), not %s" % (self.B, tuple(active.shape)))
        if active.device != self.device:
            raise ValueError("active must be on the env's device %s, not %s" % (self.device, active.device))
        return active.contiguous().view(torch.uint8)

    def step(self, actions, active=None):
        """actions: int32 CUDA tensor [B, N].  Stream-ordered, no synchronisation.  Returns the
        output buffers (obs [B,N,D] f32, reward [B,N] f32, done [B] u8, message [B] u8).

        `active`: a bool or uint8 tensor [B] on the env's device (mrb_step_masked).  Only the envs it flags are stepped;
        the state, output rows and stats of the others are left exactly as they are.  Stream-ordered and capturable
        too: the mask is read on the device when the step runs."""
        m = None if active is None else self.active_mask(active)
        if actions.device != self.device or actions.dtype != torch.int32 or not actions.is_contiguous() \
                or tuple(actions.shape) != (self.B, self.N):
            actions = actions.to(device=self.device, dtype=torch.int32).reshape(self.B, self.N).contiguous()
        with torch.cuda.device(self.device):
            if m is None:
                _lib.check(self.lib.mrb_step(self.handle, _ptr(actions), self._stream()), self.handle)
            else:
                _lib.check(self.lib.mrb_step_masked(self.handle, _ptr(actions), _ptr(m), self._stream()), self.handle)
        return self.obs, self.reward, self.done, self.message

    def host_buffers(self):
        """Pinned host mirrors used by step_host (allocated on first use)."""
        if self._host is None:
            B, N, D = self.B, self.N, self.D
            pin = dict(pin_memory=True)
            self._host = {
                "actions": torch.zeros((B, N), dtype=torch.int32, **pin),
                "obs": torch.zeros((B, N, D), dtype=torch.float32, **pin),
                "reward": torch.zeros((B, N), dtype=torch.float32, **pin),
                "done": torch.zeros((B,), dtype=torch.uint8, **pin),
                "message": torch.zeros((B,), dtype=torch.uint8, **pin),
            }
        return self._host

    def step_host(self, actions):
        """actions: host int array [B, N].  H2D actions -> step -> D2H obs/reward/done/message, one
        synchronisation at the end.  Returns the pinned host tensors."""
        h = self.host_buffers()
        a = torch.as_tensor(np.asarray(actions), dtype=torch.int32).reshape(self.B, self.N) \
            if not isinstance(actions, torch.Tensor) else actions.to(torch.int32).reshape(self.B, self.N)
        # a pinned, contiguous int32 tensor is uploaded from where it is; anything else is staged through h["actions"]
        if not (a.device.type == "cpu" and a.is_contiguous() and a.is_pinned()):
            h["actions"].copy_(a)
            a = h["actions"]
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrb_step_host(self.handle, _ptr(a), _ptr(h["obs"]), _ptr(h["reward"]),
                                              _ptr(h["done"]), _ptr(h["message"]), self._stream()), self.handle)
        return h["obs"], h["reward"], h["done"], h["message"]

    @property
    def h2d_bytes_per_step(self):
        return self.B * self.N * 4

    @property
    def d2h_bytes_per_step(self):
        return self.B * self.N * self.D * 4 + self.B * self.N * 4 + 2 * self.B

    # ------------------------------------------------------------------ state (checkpoint / parity injection)
    def _fields(self, count, names=None, source=None):
        """numpy arrays + the mrb_state_fields struct pointing at them (arrays from `source` when given)."""
        wanted = _lib.COMMON_FIELDS + _lib.SCENARIO_FIELDS[self.scenario]
        arrays, f = {}, _lib.StateFields()
        f.struct_size = C.sizeof(_lib.StateFields)
        for name, dt, shape in _lib.STATE_FIELDS:
            if name not in wanted or (names is not None and name not in names):
                continue
            full = (count,) + shape(self.N, self.P)
            if source is None:
                a = np.zeros(full, dtype=dt)
            else:
                if name not in source:
                    continue
                a = np.ascontiguousarray(np.asarray(source[name]).reshape(full), dtype=dt)
            arrays[name] = a
            setattr(f, name, a.ctypes.data)
        return arrays, f

    def get_state(self, env_lo=0, count=None, names=None):
        """Per-field state of envs [env_lo, env_lo + count) (mrb_get_state): dict of numpy arrays with a leading
        env axis, the reference's own state variables (field names and citations: include/marbler_b200.h)."""
        count = self.B - env_lo if count is None else int(count)
        arrays, f = self._fields(count, names)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrb_get_state(self.handle, int(env_lo), count, C.byref(f), self._stream()), self.handle)
        return arrays

    def set_state(self, st, env_lo=0, count=None, envs=None):
        """Overwrite the state of envs [env_lo, env_lo + count) (mrb_set_state) with the fields present in `st`
        (leading env axis); fields that are absent keep their values.  `envs`: an index array instead of a range -
        `st` then holds one entry per listed env (each env is written on its own)."""
        if envs is not None:
            envs = np.asarray(envs).reshape(-1)
            for k, e in enumerate(envs):
                self.set_state({n: np.asarray(v)[k:k + 1] for n, v in st.items()}, env_lo=int(e), count=1)
            return
        count = self.B - env_lo if count is None else int(count)
        arrays, f = self._fields(count, source=st)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrb_set_state(self.handle, int(env_lo), count, C.byref(f), self._stream()), self.handle)

    def read_stats(self, reset=False):
        v = self.stats.cpu().numpy().copy()
        if reset:
            self.stats.zero_()
        return dict(zip(_lib.STAT_NAMES, v[:len(_lib.STAT_NAMES)]))

    @property
    def agent_poses(self):
        """[B, 3, N] view-copy of the unicycle poses (the reference's scenario.agent_poses is (3, N))."""
        return self.state_f64[:3 * self.N].t().reshape(self.B, 3, self.N)


def fp64_peak(device=0, milliseconds=200.0):
    """Measured FP64 rate of independent DFMA chains on `device`, TFLOP/s (mrb_fp64_peak): the roofline the
    step kernels are compared with."""
    out = C.c_double()
    _lib.check(_lib.load().mrb_fp64_peak(int(device), float(milliseconds), C.byref(out)))
    return out.value


def barrier_qp(dxi, xi, barrier_default=False):
    """rps barrier certificate on a batch: dxi, xi CUDA f64 tensors [B, 2, N] -> (u [B, 2, N], iters [B])."""
    lib = _lib.load()
    B, _, N = dxi.shape
    dev = dxi.device
    d = dxi.permute(1, 2, 0).contiguous().to(torch.float64)
    x = xi.permute(1, 2, 0).contiguous().to(torch.float64)
    u = torch.empty_like(d)
    it = torch.zeros((B,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.mrb_barrier_qp(dev.index or 0, N, int(barrier_default), B, _ptr(d), _ptr(x), _ptr(u), _ptr(it),
                                      C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return u.permute(2, 0, 1).contiguous(), it
