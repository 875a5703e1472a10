"""Closed-loop rollouts on the device (f1l_rollout_dev): a fleet of kinematic-bicycle cars, grouped
into races whose cars are each other's opponents, advanced T planning steps by the batch planner
without leaving the GPU.

    fleet = engine.fleet(poses, group=4)       # poses [S,4] (x, y, theta, v), S % group == 0
                                               # weights=[S,5]: cost weights per car
                                               # vehicle=Vehicle(): dynamic single-track cars
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

SingleTrackTrace = namedtuple("SingleTrackTrace", RolloutTrace._fields + ("dyn",))
SingleTrackTrace.__doc__ = """Fleet.run(trace=True) of a single-track fleet: the RolloutTrace fields
and dyn [T,S,3], (steering angle, yaw rate, slip angle) at the start of step k."""

Vehicle = namedtuple("Vehicle", [f for f, _ in _lib.Vehicle._fields_],
                     defaults=(1.0489, 4.718, 5.4562, 0.15875, 0.17145, 0.074, 3.74, 0.04712, 3.2, 7.319, 0.5))
Vehicle.__doc__ = """Parameters of the dynamic single-track model (f1l_vehicle), f1tenth_gym's by
default: mu, C_Sf, C_Sr (1/rad), lf, lr, h (m), m (kg), I (kg m^2), max_steer_vel (rad/s), v_switch
and v_kin (m/s)."""


def _vehicle_struct(vehicle):
    """the f1l_vehicle of a Vehicle, ValueError for a value f1l_rollout_st_dev rejects"""
    v = Vehicle(*(float(x) for x in vehicle))
    for name, val in v._asdict().items():
        if not (val >= 0 if name == "h" else val > 0):
            raise ValueError("vehicle %s must be %s" % (name, "non-negative" if name == "h" else "positive"))
    return _lib.Vehicle(*v)


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


def _weights_tensor(weights, S, device):
    import torch
    if isinstance(weights, torch.Tensor):
        t = weights.detach()
    else:
        import numpy as np
        t = torch.from_numpy(np.array(weights, dtype=np.float64, copy=True))
    if tuple(t.shape) != (S, _lib.N_TERMS) or not t.dtype.is_floating_point:
        raise ValueError("weights must be a float array [%d, %d]" % (S, _lib.N_TERMS))
    return t.to(device=device, dtype=torch.float32).contiguous().clone()


class Fleet:
    """S cars on one Engine: state [S,4] f64, prev_theta [S,M] f32, has_prev [S] u8, status [S] u8,
    progress [S] f64, track_i [S] i32, track_s [S] f64 (f1l_fleet), all CUDA tensors on the
    engine's device.  Races are the `group` consecutive cars [g*group, (g+1)*group).  `weights` is
    a float32 CUDA tensor [S,5] of cost weights per car, or None: every car uses the engine's
    configured weights.  `vehicle` is None (kinematic bicycle) or a Vehicle: the cars follow the
    dynamic single-track model and the fleet also owns dyn [S,3] f64, each car's (steering angle,
    yaw rate, slip angle), zeros at creation."""

    def __init__(self, engine, poses, group=1, weights=None, vehicle=None):
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
        self.weights = None if weights is None else _weights_tensor(weights, S, dev)
        self.vehicle = None
        self.dyn = None
        if vehicle is not None:
            self.vehicle = Vehicle(*vehicle)
            _vehicle_struct(self.vehicle)   # a bad value fails here rather than at run()
            self.dyn = torch.zeros(S, 3, dtype=torch.float64, device=dev)

    @property
    def n_cars(self):
        return self.state.shape[0]

    def _buffers(self):
        dims, dev = {"S": self.n_cars, "M": self.engine.n_samples}, self.engine.device
        for name, row in _lib.FLEET_FIELDS.items():
            _lib.check_array("fleet " + name, getattr(self, name), _lib.shape_of(row, dims), row[0], dev)
        if self.weights is not None:   # read as a batch call's weights
            row = _lib.BATCH_FIELDS["weights"]
            _lib.check_array("fleet weights", self.weights, _lib.shape_of(row, dims), row[0], dev)
        if self.vehicle is not None:
            row = _lib.ST_FIELDS["dyn"]
            _lib.check_array("fleet dyn", self.dyn, _lib.shape_of(row, dims), row[0], dev)
        return _lib.FleetBuffers(**{name: getattr(self, name).data_ptr() for name in _lib.FLEET_FIELDS})

    def run(self, n_steps, dt=0.01, substeps=1, max_steer=0.4189, max_accel=9.51, v_max=math.inf,
            trace=False, stream=None, predict=False, v_min=1.0):
        """Advance every car n_steps planning steps on `stream` (default: torch's current stream)
        without synchronising.  Returns a RolloutTrace (SingleTrackTrace for a fleet with a
        vehicle) of CUDA tensors with trace=True, else None.  predict=True: every planner sees its
        opponents moving at their current velocity (along the heading, for single-track cars along
        the course psi + slip angle; frozen cars stand) and times itself at max(v, v_min)
        (f1l_rollout_predict_dev)."""
        import torch
        n_steps = int(n_steps)
        if n_steps < 0:
            raise ValueError("n_steps must be >= 0")
        if int(substeps) < 1:
            raise ValueError("substeps must be >= 1")
        for name, val in (("dt", dt), ("max_steer", max_steer), ("max_accel", max_accel), ("v_max", v_max)):
            if not float(val) > 0:
                raise ValueError("%s must be positive" % name)
        if predict and not (math.isfinite(float(v_min)) and float(v_min) > 0):
            raise ValueError("v_min must be finite and positive")
        rc = _lib.RolloutConfig(float(dt), int(substeps), self.group, float(max_steer), float(max_accel),
                                float(v_max))
        veh = _vehicle_struct(self.vehicle) if self.vehicle is not None else None
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
            if veh is not None:
                out = SingleTrackTrace(*out, torch.empty(n_steps, S, 3, dtype=torch.float64, device=dev))
        st = stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream
        eng = self.engine
        w = C.c_void_p(self.weights.data_ptr() if self.weights is not None else None)
        tbp = C.byref(tb) if tb is not None else None
        if predict:
            eng._ck(eng._L.f1l_rollout_predict_dev(
                eng._h, C.byref(rc), C.byref(veh) if veh is not None else None, C.byref(fl),
                C.c_void_p(self.dyn.data_ptr() if veh is not None else None), w, float(v_min), S, n_steps, tbp,
                C.c_void_p(out.dyn.data_ptr() if trace and veh is not None else None), C.c_void_p(st)))
        elif veh is None:
            eng._ck(eng._L.f1l_rollout_weights_dev(eng._h, C.byref(rc), C.byref(fl), w, S, n_steps, tbp,
                                                   C.c_void_p(st)))
        else:
            eng._ck(eng._L.f1l_rollout_st_dev(eng._h, C.byref(rc), C.byref(veh), C.byref(fl),
                                              C.c_void_p(self.dyn.data_ptr()), w, S, n_steps, tbp,
                                              C.c_void_p(out.dyn.data_ptr() if trace else None),
                                              C.c_void_p(st)))
        return out

    def reset(self, cars, poses):
        """Put `cars` (indices) back on the road at `poses` [n,4] as fresh cars: no previous path,
        status 0, progress 0, raceline tracking re-acquired on the next run(), and with a vehicle
        dyn 0 (straight wheels, no yaw rate, no slip).  Their weights stay."""
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
        if self.dyn is not None:
            self.dyn[idx] = 0.0
