"""Closed-loop rollouts on the device (f1l_rollout_dev): a fleet of kinematic-bicycle cars, grouped
into races whose cars are each other's opponents, advanced T planning steps by the batch planner
without leaving the GPU.

    fleet = engine.fleet(poses, group=4)       # poses [S,4] (x, y, theta, v), S % group == 0
    tr = fleet.run(500, substeps=5, trace=True)
    fleet.status, fleet.progress               # F1L_CAR_* bits, metres along the raceline

Every buffer of the fleet is a CUDA tensor the library reads and writes in place, so consecutive
run() calls continue where the last one stopped.
"""
import ctypes as C
import math
from collections import namedtuple

from . import _lib
from ._lib import CAR_HIT_MAP, CAR_HIT_CAR, CAR_NO_FEASIBLE, MAX_GROUP  # noqa: F401

RolloutTrace = namedtuple("RolloutTrace", ["state", "steer_speed", "best_idx", "status", "progress"])
RolloutTrace.__doc__ = """Per-step record of Fleet.run(trace=True): state [T,S,4] at the start of
step k, steer_speed [T,S,2] the raw planner command, best_idx [T,S], status [T,S] and progress [T,S]
after step k."""


def _poses_tensor(poses, device):
    import torch
    if isinstance(poses, torch.Tensor):
        t = poses.detach()
    else:
        import numpy as np
        t = torch.from_numpy(np.array(poses, dtype=np.float64, copy=True))
    if t.ndim != 2 or t.shape[1] != 4 or not t.dtype.is_floating_point:
        raise ValueError("poses must be a float array [S, 4] (x, y, theta, v)")
    return t.to(device=device, dtype=torch.float64).contiguous().clone()   # the fleet owns its state


class Fleet:
    """S cars on one Engine: state [S,4] f64, prev_theta [S,M] f32, has_prev [S] u8, status [S] u8,
    progress [S] f64, track_i [S] i32, track_s [S] f64 (f1l_fleet), all CUDA tensors on the
    engine's device.  Races are the `group` consecutive cars [g*group, (g+1)*group)."""

    def __init__(self, engine, poses, group=1):
        import torch
        group = int(group)
        dev = torch.device("cuda", engine.device)
        state = _poses_tensor(poses, dev)
        S = state.shape[0]
        if not 1 <= group <= MAX_GROUP:
            raise ValueError("group must be in 1..%d" % MAX_GROUP)
        if S == 0 or S % group:
            raise ValueError("the number of cars (%d) must be a positive multiple of group (%d)" % (S, group))
        self.engine = engine
        self.group = group
        self.state = state
        self.prev_theta = torch.zeros(S, engine.n_samples, dtype=torch.float32, device=dev)
        self.has_prev = torch.zeros(S, dtype=torch.uint8, device=dev)
        self.status = torch.zeros(S, dtype=torch.uint8, device=dev)
        self.progress = torch.zeros(S, dtype=torch.float64, device=dev)
        self.track_i = torch.full((S,), -1, dtype=torch.int32, device=dev)
        self.track_s = torch.zeros(S, dtype=torch.float64, device=dev)

    @property
    def n_cars(self):
        return self.state.shape[0]

    def _buffers(self):
        for name, dtype, shape in (("state", "float64", (self.n_cars, 4)),
                                   ("prev_theta", "float32", (self.n_cars, self.engine.n_samples)),
                                   ("has_prev", "uint8", (self.n_cars,)), ("status", "uint8", (self.n_cars,)),
                                   ("progress", "float64", (self.n_cars,)), ("track_i", "int32", (self.n_cars,)),
                                   ("track_s", "float64", (self.n_cars,))):
            t = getattr(self, name)
            if (not t.is_cuda or t.device.index != self.engine.device or str(t.dtype) != "torch." + dtype
                    or tuple(t.shape) != shape or not t.is_contiguous()):
                raise ValueError("fleet buffer %s must be a contiguous %s CUDA tensor %s on cuda:%d"
                                 % (name, dtype, list(shape), self.engine.device))
        return _lib.FleetBuffers(*(t.data_ptr() for t in (
            self.state, self.prev_theta, self.has_prev, self.status, self.progress, self.track_i,
            self.track_s)))

    def run(self, n_steps, dt=0.01, substeps=1, max_steer=0.4189, max_accel=9.51, v_max=math.inf,
            trace=False, stream=None):
        """Advance every car n_steps planning steps on `stream` (default: torch's current stream)
        without synchronising.  Returns a RolloutTrace of CUDA tensors with trace=True, else None."""
        import torch
        n_steps = int(n_steps)
        if n_steps < 0:
            raise ValueError("n_steps must be >= 0")
        if int(substeps) < 1:
            raise ValueError("substeps must be >= 1")
        for name, val in (("dt", dt), ("max_steer", max_steer), ("max_accel", max_accel), ("v_max", v_max)):
            if not float(val) > 0:
                raise ValueError("%s must be positive" % name)
        rc = _lib.RolloutConfig(float(dt), int(substeps), self.group, float(max_steer), float(max_accel),
                                float(v_max))
        fl = self._buffers()
        S, dev = self.n_cars, self.state.device
        out = None
        tb = None
        if trace:
            out = RolloutTrace(torch.empty(n_steps, S, 4, dtype=torch.float64, device=dev),
                               torch.empty(n_steps, S, 2, dtype=torch.float64, device=dev),
                               torch.empty(n_steps, S, dtype=torch.int32, device=dev),
                               torch.empty(n_steps, S, dtype=torch.uint8, device=dev),
                               torch.empty(n_steps, S, dtype=torch.float64, device=dev))
            tb = _lib.RolloutTraceBuffers(*(t.data_ptr() for t in out))
        st = stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream
        eng = self.engine
        eng._ck(eng._L.f1l_rollout_dev(eng._h, C.byref(rc), C.byref(fl), S, n_steps,
                                       C.byref(tb) if tb is not None else None, C.c_void_p(st)))
        return out

    def reset(self, cars, poses):
        """Put `cars` (indices) back on the road at `poses` [n,4] as fresh cars: no previous path,
        status 0, progress 0, raceline tracking re-acquired on the next run()."""
        import torch
        idx = torch.as_tensor(cars, dtype=torch.long).reshape(-1).to(self.state.device)
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= self.n_cars):
            raise ValueError("car index out of range")
        p = _poses_tensor(poses, self.state.device)
        if p.shape[0] != idx.numel():
            raise ValueError("one pose per reset car")
        self.state[idx] = p
        self.has_prev[idx] = 0
        self.status[idx] = 0
        self.progress[idx] = 0.0
        self.track_i[idx] = -1
