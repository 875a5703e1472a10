"""Engine: one per-device planner handle of the C-ABI library (include/f1l.h).

This is the thin host layer the reference-shaped classes (lattice_planner.LatticePlanner,
pure_pursuit.PurePursuitPlanner, utils.*) sit on.  numpy arrays carry host buffers, torch
tensors carry device buffers for the ``*_dev`` calls; no arithmetic of the hot path happens here.
"""
import ctypes as C
import os
from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import (N_TERMS, MAX_OPP, FLAG_VALID, FLAG_COLLIDE_OPP, FLAG_COLLIDE_MAP,  # noqa: F401
                   FLAG_NO_CENTRE, F1LError)

_dp, _fp, _ip, _bp = _lib._dp, _lib._fp, _lib._ip, _lib._bp

PlanDetail = namedtuple("PlanDetail", [
    "steer", "speed", "best_traj", "best_idx", "best_cost", "costs", "terms", "flags", "goals",
    "params", "states", "no_feasible", "tracker_found", "headings", "best_traj_map"],
    defaults=[None])

BatchPlan = namedtuple("BatchPlan", ["best_idx", "best_cost", "best_traj", "costs", "flags",
                                     "steer_speed"])

PurePursuitBatch = namedtuple("PurePursuitBatch", ["nearest", "nearest_i", "lookahead",
                                                   "lookahead_i", "actuation", "status"])


def default_device():
    return int(os.environ.get("LOCAL_RANK", "0"))


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a, typ):
    return a.ctypes.data_as(typ) if a is not None else typ()


def _vp(a):
    """void* of a numpy array / torch tensor / None."""
    if a is None:
        return C.c_void_p()
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(a.data_ptr())


class Engine:
    """Owns an f1l_handle.  Config keywords are the fields of f1l_config (include/f1l.h)."""

    def __init__(self, device=None, **config):
        self._h = C.c_void_p()
        self._L = _lib.lib()
        cfg = _lib.default_config()
        self._apply(cfg, config)
        dev = default_device() if device is None else int(device)
        _lib.check(self._L.f1l_create(C.byref(self._h), dev, C.byref(cfg)))
        self._n_samples = int(cfg.n_samples)
        self.device = dev
        self.n_lookaheads = 0
        self.n_widths = 0
        self.n_waypoints = 0
        self.peer_world = 0

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.f1l_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, code):
        _lib.check(code, self._h)

    # -- configuration ----------------------------------------------------------------------
    @staticmethod
    def _apply(cfg, kw):
        for k, v in kw.items():
            if k == "weights":
                if len(v) != N_TERMS:
                    raise ValueError("weights must have %d entries" % N_TERMS)
                for i, w in enumerate(v):
                    cfg.weights[i] = float(w)
            elif hasattr(cfg, k):
                setattr(cfg, k, v)
            else:
                raise TypeError("unknown config field %r" % k)

    @property
    def config(self):
        cfg = _lib.Config()
        self._ck(self._L.f1l_get_config(self._h, C.byref(cfg)))
        return cfg

    def configure(self, **kw):
        cfg = self.config
        self._apply(cfg, kw)
        self._ck(self._L.f1l_set_config(self._h, C.byref(cfg)))
        self._n_samples = int(cfg.n_samples)

    @property
    def n_candidates(self):
        return self.n_lookaheads * self.n_widths

    # -- uploads ----------------------------------------------------------------------------
    def set_track(self, waypoints):
        w = _f64(waypoints)
        if w.ndim != 2 or w.shape[1] < 2 or w.shape[0] < 2:
            raise ValueError("waypoints must be [N>=2, ncols>=2]")
        self._ck(self._L.f1l_set_track(self._h, _ptr(w, _dp), w.shape[0], w.shape[1]))
        self.n_waypoints = w.shape[0]

    def set_grid(self, occ, origin, resolution):
        g = np.ascontiguousarray(occ, dtype=np.uint8)
        self._ck(self._L.f1l_set_grid(self._h, _ptr(g, _bp), g.shape[0], g.shape[1],
                                      float(origin[0]), float(origin[1]), float(resolution)))

    def get_edt(self, shape):
        """[H, W] uint16 squared cell distance to the nearest occupied / out-of-bounds cell (exact
        to 576, 577 = farther): the transform collision_mode=1 looks up (f1l_get_edt)."""
        out = np.zeros(shape, np.uint16)
        self._ck(self._L.f1l_get_edt(self._h, _vp(out)))
        return out

    def clear_grid(self):
        self._ck(self._L.f1l_clear_grid(self._h))

    def set_goal_grid(self, lookaheads, widths):
        la, wd = _f64(lookaheads).ravel(), _f64(widths).ravel()
        self._ck(self._L.f1l_set_goal_grid(self._h, _ptr(la, _dp), la.size, _ptr(wd, _dp), wd.size))
        self.n_lookaheads, self.n_widths = la.size, wd.size

    def get_lut(self):
        dims = (C.c_int32 * 3)()
        rng = (C.c_double * 6)()
        self._ck(self._L.f1l_get_lut_shape(self._h, dims, rng))
        out = np.zeros((dims[0], dims[1], dims[2], 4), dtype=np.float32)
        self._ck(self._L.f1l_get_lut(self._h, _ptr(out, _fp)))
        return out, tuple(rng)

    def set_lut(self, lut, ranges):
        lut = np.ascontiguousarray(lut, dtype=np.float32)
        dims = (C.c_int32 * 3)(*lut.shape[:3])
        rng = (C.c_double * 6)(*[float(r) for r in ranges])
        self._ck(self._L.f1l_set_lut(self._h, _ptr(lut, _fp), dims, rng))

    def set_prev_path(self, theta_prev):
        if theta_prev is None:
            self._ck(self._L.f1l_clear_prev_path(self._h))
            return
        t = np.ascontiguousarray(theta_prev, dtype=np.float32)
        self._ck(self._L.f1l_set_prev_path(self._h, _ptr(t, _fp), t.size))

    # -- single query -----------------------------------------------------------------------
    def _result(self, C_, detail, want_states, want_headings=False, want_map=False):
        M = self.n_samples
        res = _lib.PlanResult()
        bufs = {"best_traj": np.empty((M, 4), np.float32)}
        res.best_traj = bufs["best_traj"].ctypes.data
        if want_map:
            bufs["best_traj_map"] = np.empty((M, 4), np.float64)
            res.best_traj_map = bufs["best_traj_map"].ctypes.data
        if detail:
            bufs["costs"] = np.empty(C_, np.float32)
            bufs["terms"] = np.empty((C_, N_TERMS), np.float32)
            bufs["flags"] = np.empty(C_, np.uint8)
            bufs["goals"] = np.empty((C_, 3), np.float32)
            bufs["params"] = np.empty((C_, 4), np.float32)
            res.costs = bufs["costs"].ctypes.data
            res.terms = bufs["terms"].ctypes.data
            res.flags = bufs["flags"].ctypes.data
            res.goals = bufs["goals"].ctypes.data
            res.params = bufs["params"].ctypes.data
        if want_states:
            bufs["states"] = np.zeros((C_, M, 4), np.float32)
            res.states = bufs["states"].ctypes.data
        if want_headings:
            bufs["headings"] = np.zeros((C_, M, 2), np.float32)
            res.headings = bufs["headings"].ctypes.data
        return res, bufs

    @staticmethod
    def _detail(res, bufs):
        return PlanDetail(res.steer, res.speed, bufs["best_traj"], res.best_idx, res.best_cost,
                          bufs.get("costs"), bufs.get("terms"), bufs.get("flags"),
                          bufs.get("goals"), bufs.get("params"), bufs.get("states"),
                          bool(res.no_feasible), bool(res.tracker_found), bufs.get("headings"),
                          bufs.get("best_traj_map"))

    @staticmethod
    def _opp(opponent_poses):
        if opponent_poses is None:
            return None, 0
        o = _f64(opponent_poses).reshape(-1, 3)
        if o.shape[0] > MAX_OPP:
            raise ValueError("at most %d opponents" % MAX_OPP)
        return (o, o.shape[0]) if o.shape[0] else (None, 0)

    @property
    def n_samples(self):
        return self._n_samples

    def plan(self, pose, opponent_poses=None, update_prev=True, detail=True, want_states=False,
             shard=None, want_headings=False, rows=None, want_map=False):
        """One query.  pose = (x, y, theta, velocity).  Dense-sweep sharding across GPUs:
        shard = (c_begin, c_end) evaluates a candidate range only, rows = (row_begin, row_step)
        the lookahead rows row_begin, row_begin + row_step, ... (balanced across ranks).  With
        attach_peers() both are collective and return the global winner on every rank (and
        rows= then honours update_prev: every rank stores the same previous path)."""
        pose = _f64(pose).ravel()
        if pose.size != 4:
            raise ValueError("pose must be (x, y, theta, velocity)")
        opp, k = self._opp(opponent_poses)
        res, bufs = self._result(self.n_candidates, detail, want_states, want_headings, want_map)
        if rows is not None:
            code = self._L.f1l_plan_rows(self._h, pose.ctypes.data, opp.ctypes.data if k else None,
                                         k, int(rows[0]), int(rows[1]),
                                         int(bool(update_prev) and self.peer_world > 1), C.byref(res))
        elif shard is None:
            code = self._L.f1l_plan(self._h, pose.ctypes.data, opp.ctypes.data if k else None, k,
                                    int(bool(update_prev)), C.byref(res))
        else:
            code = self._L.f1l_plan_shard(self._h, pose.ctypes.data, opp.ctypes.data if k else None,
                                          k, int(shard[0]), int(shard[1]), C.byref(res))
        self._ck(code)
        return self._detail(res, bufs)

    def plan_goals(self, pose, goals, opponent_poses=None, update_prev=True, detail=True,
                   want_states=False, want_map=False):
        pose = _f64(pose).ravel()
        g = _f64(goals).reshape(-1, 3)
        opp, k = self._opp(opponent_poses)
        res, bufs = self._result(g.shape[0], detail, want_states, want_map=want_map)
        self._ck(self._L.f1l_plan_goals(self._h, pose.ctypes.data, g.ctypes.data, g.shape[0],
                                        opp.ctypes.data if k else None, k, int(bool(update_prev)),
                                        C.byref(res)))
        return self._detail(res, bufs)

    def select_candidate(self, idx, cost=0.0, update_prev=True, want_map=False):
        """Tracker output and trajectory of candidate `idx` of the last plan() / plan_goals() query
        (a selection made by user code, f1l_select_candidate) -> PlanDetail without the
        per-candidate arrays."""
        res, bufs = self._result(0, False, False, want_map=want_map)
        self._ck(self._L.f1l_select_candidate(self._h, int(idx), float(cost), int(bool(update_prev)),
                                              C.byref(res)))
        return self._detail(res, bufs)

    def generate(self, goals):
        """goals [C,3] -> (states [C,M,4], params [C,4], valid [C])."""
        g = _f64(goals).reshape(-1, 3)
        M = self.n_samples
        states = np.zeros((g.shape[0], M, 4), np.float32)
        params = np.zeros((g.shape[0], 4), np.float32)
        flags = np.zeros(g.shape[0], np.uint8)
        if g.shape[0] == 0:
            return states, params, flags != 0
        self._ck(self._L.f1l_generate(self._h, _ptr(g, _dp), g.shape[0], _ptr(states, _fp),
                                      _ptr(params, _fp), _ptr(flags, _bp)))
        return states, params, (flags & FLAG_VALID) != 0

    # -- batch ------------------------------------------------------------------------------
    def _check_prev(self, S, prev_theta, has_prev, update_prev, is_dev):
        """Validates the per-scenario previous paths of plan_batch / plan_batch_dev.  They are
        read and, with update_prev, written in place, so anything that would need a copy (wrong
        type, shape, dtype, layout or device) is a ValueError rather than a silent conversion."""
        if prev_theta is None:
            if has_prev is not None or update_prev:
                raise ValueError("has_prev / update_prev need prev_theta")
            return
        shape = (S, self.n_samples)
        if is_dev:
            import torch
            ok_type = isinstance(prev_theta, torch.Tensor) and prev_theta.is_cuda
            if not (ok_type and prev_theta.dtype == torch.float32 and tuple(prev_theta.shape) == shape
                    and prev_theta.is_contiguous() and prev_theta.device.index == self.device):
                raise ValueError("prev_theta must be a contiguous float32 CUDA tensor [%d, %d] on "
                                 "cuda:%d" % (S, self.n_samples, self.device))
            if has_prev is not None and not (
                    isinstance(has_prev, torch.Tensor) and has_prev.is_cuda
                    and has_prev.dtype in (torch.uint8, torch.bool) and tuple(has_prev.shape) == (S,)
                    and has_prev.is_contiguous() and has_prev.device == prev_theta.device):
                raise ValueError("has_prev must be a contiguous uint8 / bool CUDA tensor [%d] on "
                                 "prev_theta's device" % S)
            return
        if not (isinstance(prev_theta, np.ndarray) and prev_theta.dtype == np.float32
                and prev_theta.shape == shape and prev_theta.flags.c_contiguous):
            raise ValueError("prev_theta must be a C-contiguous float32 numpy array [%d, %d]"
                             % (S, self.n_samples))
        if has_prev is not None and not (
                isinstance(has_prev, np.ndarray) and has_prev.dtype in (np.uint8, np.bool_)
                and has_prev.shape == (S,) and has_prev.flags.c_contiguous):
            raise ValueError("has_prev must be a contiguous uint8 / bool numpy array [%d]" % S)
        if update_prev and not (prev_theta.flags.writeable
                                and (has_prev is None or has_prev.flags.writeable)):
            raise ValueError("update_prev writes prev_theta / has_prev in place: they must be writeable")

    def plan_batch(self, poses, opponents=None, n_opp=None, out=None, want_traj=True,
                   want_costs=True, want_flags=False, prev_theta=None, has_prev=None,
                   update_prev=False):
        """S independent scenarios with HOST buffers (numpy; pinned if allocated through
        ``pinned_empty``).  poses [S,4], opponents [S,K,3], n_opp [S].

        Previous paths of the similarity cost, one per scenario (f1l_plan_batch_prev):
        prev_theta [S, n_samples] C-contiguous float32, the theta column of each scenario's
        previous best trajectory; has_prev [S] bool / uint8 (None: every scenario has one).
        Scenario s then plans exactly as plan() after set_prev_path(prev_theta[s]) (or
        set_prev_path(None) where has_prev[s] is 0).  update_prev=True overwrites both arrays in
        place with this call's best trajectories' theta columns and ones, ready for the next
        step.  The engine's own previous path (set_prev_path) is not used."""
        poses = _f64(poses).reshape(-1, 4)
        S = poses.shape[0]
        self._check_prev(S, prev_theta, has_prev, update_prev, False)
        K = 0
        if opponents is not None:
            opponents = _f64(opponents)
            K = opponents.shape[1]
        if n_opp is not None:
            n_opp = np.ascontiguousarray(n_opp, dtype=np.int32)
        Cn, M = self.n_candidates, self.n_samples
        o = out or {}
        best_idx = o.get("best_idx", None)
        if best_idx is None:
            best_idx = np.zeros(S, np.int32)
        best_cost = o.get("best_cost") if o.get("best_cost") is not None else np.zeros(S, np.float32)
        steer_speed = (o.get("steer_speed") if o.get("steer_speed") is not None
                       else np.zeros((S, 2), np.float64))
        best_traj = o.get("best_traj") if want_traj else None
        if want_traj and best_traj is None:
            best_traj = np.zeros((S, M, 4), np.float32)
        costs = o.get("costs") if want_costs else None
        if want_costs and costs is None:
            costs = np.zeros((S, Cn), np.float32)
        flags = o.get("flags") if want_flags else None
        if want_flags and flags is None:
            flags = np.zeros((S, Cn), np.uint8)
        if S == 0:   # an empty batch is a valid (empty) answer, not an error
            return BatchPlan(best_idx, best_cost, best_traj, costs, flags, steer_speed)
        if prev_theta is None:
            self._ck(self._L.f1l_plan_batch(self._h, _vp(poses), _vp(opponents), _vp(n_opp), S, K,
                                            _vp(best_idx), _vp(best_cost), _vp(best_traj),
                                            _vp(costs), _vp(flags), _vp(steer_speed)))
        else:
            self._ck(self._L.f1l_plan_batch_prev(self._h, _vp(poses), _vp(opponents), _vp(n_opp),
                                                 S, K, _vp(prev_theta), _vp(has_prev),
                                                 int(bool(update_prev)), _vp(best_idx),
                                                 _vp(best_cost), _vp(best_traj), _vp(costs),
                                                 _vp(flags), _vp(steer_speed)))
        return BatchPlan(best_idx, best_cost, best_traj, costs, flags, steer_speed)

    def plan_batch_dev(self, poses, opponents=None, n_opp=None, best_idx=None, best_cost=None,
                       best_traj=None, costs=None, flags=None, steer_speed=None, stream=None,
                       prev_theta=None, has_prev=None, update_prev=False):
        """Same with torch CUDA tensors; enqueues on `stream` (default: torch's current stream)
        and does not synchronise.  prev_theta / has_prev / update_prev as for plan_batch, as
        contiguous CUDA tensors (float32 [S, n_samples], uint8 / bool [S]) updated in place on
        the stream (f1l_plan_batch_prev_dev)."""
        import torch
        S = poses.shape[0]
        K = 0 if opponents is None else opponents.shape[1]
        self._check_prev(S, prev_theta, has_prev, update_prev, True)
        st = stream if stream is not None else torch.cuda.current_stream(poses.device).cuda_stream
        if prev_theta is None:
            self._ck(self._L.f1l_plan_batch_dev(self._h, _vp(poses), _vp(opponents), _vp(n_opp), S,
                                                K, _vp(best_idx), _vp(best_cost), _vp(best_traj),
                                                _vp(costs), _vp(flags), _vp(steer_speed),
                                                C.c_void_p(st)))
        else:
            self._ck(self._L.f1l_plan_batch_prev_dev(self._h, _vp(poses), _vp(opponents),
                                                     _vp(n_opp), S, K, _vp(prev_theta),
                                                     _vp(has_prev), int(bool(update_prev)),
                                                     _vp(best_idx), _vp(best_cost),
                                                     _vp(best_traj), _vp(costs), _vp(flags),
                                                     _vp(steer_speed), C.c_void_p(st)))

    # -- closed-loop rollouts ----------------------------------------------------------------
    def fleet(self, poses, group=1):
        """A fleet of kinematic-bicycle cars at `poses` [S,4] (x, y, theta, v) on this engine's
        device, raced in groups of `group` consecutive cars (rollout.Fleet, f1l_rollout_dev)."""
        from .rollout import Fleet
        return Fleet(self, poses, group)

    # -- candidate sharding over peer memory -------------------------------------------------
    def export_peer_handle(self):
        """64-byte CUDA IPC handle of this engine's exchange block (f1l_xchg_export)."""
        buf = (C.c_uint8 * 64)()
        self._ck(self._L.f1l_xchg_export(self._h, buf, 64))
        return bytes(buf)

    def attach_peer_handles(self, rank, handles):
        """handles: the export_peer_handle() bytes of every rank, in rank order (f1l_xchg_attach).
        Afterwards plan(shard=...) is collective and returns the global winner on every rank."""
        world = len(handles)
        blob = (C.c_uint8 * (64 * world)).from_buffer_copy(b"".join(handles))
        self._ck(self._L.f1l_xchg_attach(self._h, int(rank), world, blob))
        self.peer_world = world

    def attach_peers(self, group=None):
        """Exchange the IPC handles over torch.distributed (any backend) and attach; collective."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        handles = [None] * world
        dist.all_gather_object(handles, self.export_peer_handle(), group=group)
        self.attach_peer_handles(rank, handles)
        dist.barrier(group=group)   # nobody starts a collective query before everybody is attached

    def detach_peers(self, group=None):
        if group is not False:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dist.barrier(group=group)   # nobody unmaps a block a peer may still write
        self._ck(self._L.f1l_xchg_detach(self._h))
        self.peer_world = 0

    # -- pure pursuit -----------------------------------------------------------------------
    def pure_pursuit_batch(self, poses, lookahead_distance, out=None):
        """B poses [B,3] (x, y, theta), HOST buffers -> PurePursuitBatch of numpy arrays."""
        poses = _f64(poses).reshape(-1, 3)
        B = poses.shape[0]
        o = out or {}
        nearest = o.get("nearest") if o.get("nearest") is not None else np.zeros((B, 4))
        nearest_i = o.get("nearest_i") if o.get("nearest_i") is not None else np.zeros(B, np.int32)
        look = o.get("lookahead") if o.get("lookahead") is not None else np.zeros((B, 4))
        look_i = o.get("lookahead_i") if o.get("lookahead_i") is not None else np.zeros(B, np.int32)
        act = o.get("actuation") if o.get("actuation") is not None else np.zeros((B, 2))
        status = o.get("status") if o.get("status") is not None else np.zeros(B, np.int32)
        if B == 0:
            return PurePursuitBatch(nearest, nearest_i, look, look_i, act, status)
        self._ck(self._L.f1l_pure_pursuit_batch(self._h, _vp(poses), B, float(lookahead_distance),
                                                _vp(nearest), _vp(nearest_i), _vp(look),
                                                _vp(look_i), _vp(act), _vp(status)))
        return PurePursuitBatch(nearest, nearest_i, look, look_i, act, status)

    def pure_pursuit_batch_dev(self, poses, lookahead_distance, nearest=None, nearest_i=None,
                               lookahead=None, lookahead_i=None, actuation=None, status=None,
                               stream=None):
        import torch
        st = stream if stream is not None else torch.cuda.current_stream(poses.device).cuda_stream
        self._ck(self._L.f1l_pure_pursuit_batch_dev(
            self._h, _vp(poses), poses.shape[0], float(lookahead_distance), _vp(nearest),
            _vp(nearest_i), _vp(lookahead), _vp(lookahead_i), _vp(actuation), _vp(status),
            C.c_void_p(st)))

    def front_axle_batch(self, states, wheelbase, k_path=5.0):
        """states [B,4] (x, y, theta, velocity) -> (front [B,6], target_index [B]); front columns:
        theta_e, ef, theta_raceline, kappa_ref, goal_velocity, Stanley delta."""
        st = _f64(states).reshape(-1, 4)
        front = np.zeros((st.shape[0], 6))
        idx = np.zeros(st.shape[0], np.int32)
        if st.shape[0] == 0:
            return front, idx
        self._ck(self._L.f1l_front_axle_batch(self._h, _vp(st), st.shape[0], float(wheelbase),
                                              float(k_path), _vp(front), _vp(idx)))
        return front, idx

    def intersect_point_batch(self, points, t_start, radius, wrap):
        pts = _f64(points).reshape(-1, 2)
        t0 = _f64(t_start).ravel()
        n = pts.shape[0]
        out = np.zeros((n, 4))
        out_i = np.zeros(n, np.int32)
        if n == 0:
            return out, out_i
        self._ck(self._L.f1l_intersect_point_batch(self._h, _ptr(pts, _dp), _ptr(t0, _dp), n,
                                                   float(radius), int(bool(wrap)), _ptr(out, _dp),
                                                   _ptr(out_i, _ip)))
        return out, out_i

    def get_actuation_batch(self, rows, wheelbase):
        rows = _f64(rows).reshape(-1, 7)
        out = np.zeros((rows.shape[0], 2))
        self._ck(self._L.f1l_get_actuation_batch(self._h, _ptr(rows, _dp), rows.shape[0],
                                                 float(wheelbase), _ptr(out, _dp)))
        return out

    # -- evidence ---------------------------------------------------------------------------
    @property
    def launch_count(self):
        return int(self._L.f1l_launch_count(self._h))

    def set_stats(self, on):
        """collect the deviation-pass work counters (off by default, f1l_set_stats)"""
        self._ck(self._L.f1l_set_stats(self._h, int(bool(on))))

    def stats(self):
        """(segment_steps, candidates) of the raceline-deviation pass since the last call (while
        set_stats(True)): the
        (candidate, window segment) pairs evaluated and the valid candidates that reached the
        pass.  Resets the counters (f1l_get_stats)."""
        out = (C.c_uint64 * 2)()
        self._ck(self._L.f1l_get_stats(self._h, out, 2))
        return int(out[0]), int(out[1])

    def last_eval_shape(self):
        """Template instance and CTA plan of the last eval_kernel launch (f1l_last_eval_shape):
        dict with ipl, s, sg, nw, minb, chunk, ctas_per_scenario, item and the instance `name`."""
        out = (C.c_int32 * 8)()
        self._ck(self._L.f1l_last_eval_shape(self._h, out, 8))
        keys = ("ipl", "s", "sg", "nw", "minb", "chunk", "ctas_per_scenario", "item")
        d = {k: int(v) for k, v in zip(keys, out)}
        d["name"] = "eval_kernel<%d,%d,%d,%d,%d>" % tuple(out[:5])
        return d

    def set_graph(self, on):
        """replay the single-query chain as a CUDA graph (default on)"""
        self._ck(self._L.f1l_set_graph(self._h, int(bool(on))))

    def set_timing(self, on):
        self._ck(self._L.f1l_set_timing(self._h, int(bool(on))))

    def last_kernel_ms(self):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        self._ck(self._L.f1l_last_kernel_ms(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def mean_kernel_ms(self):
        """(sample, eval, select, n): mean device ms per kernel over the launches recorded since
        set_timing(True) (most recent 64)."""
        a, b, c, n = C.c_float(), C.c_float(), C.c_float(), C.c_int()
        self._ck(self._L.f1l_mean_kernel_ms(self._h, C.byref(a), C.byref(b), C.byref(c),
                                            C.byref(n)))
        return a.value, b.value, c.value, n.value

    def measure_peaks(self):
        """(FP32 FMA TFLOP/s, MUFU Gop/s) measured on this device."""
        a, b = C.c_double(), C.c_double()
        self._ck(self._L.f1l_measure_peaks(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def measure_peaks_ex(self):
        """dict: ffma_tflops, mufu_gops, ffma2_tflops (packed fma.rn.f32x2), mixed_ipc_per_sm"""
        out = np.zeros(4)
        self._ck(self._L.f1l_measure_peaks_ex(self._h, _ptr(out, _dp), 4))
        return dict(ffma_tflops=out[0], mufu_gops=out[1], ffma2_tflops=out[2],
                    mixed_ipc_per_sm=out[3])

    def debug_query_ctx(self):
        f = np.zeros(8 + 4 * MAX_OPP, np.float32)
        i = np.zeros(6, np.int32)
        self._ck(self._L.f1l_debug_query_ctx(self._h, _ptr(f, _fp), _ptr(i, _ip)))
        return f, i


_fp_weights = {}


def fingerprint(arr):
    """(shape, 64-bit multilinear hash) of a float64 array: sum of (bit pattern x odd random
    weight) mod 2^64 over EVERY element, so any in-place edit of any row changes it (a single
    changed element always does: odd weights are invertible mod 2^64).  ~8 us for a 2000 x 5
    raceline, against ~50 us for zlib.crc32 over the same bytes -- cheap enough to run on every
    plan() call, which is what detects an edited raceline."""
    a = np.ascontiguousarray(arr, dtype=np.float64)
    v = a.reshape(-1).view(np.uint64)
    w = _fp_weights.get(v.size)
    if w is None:
        w = np.random.default_rng(0x5eed + v.size).integers(0, 2 ** 63, size=v.size, dtype=np.uint64)
        w = w * np.uint64(2) + np.uint64(1)
        _fp_weights[v.size] = w
    return a.shape, int(np.dot(v, w))


def pinned_empty(shape, dtype):
    """numpy view of a pinned host buffer (torch is only the allocator)."""
    import torch
    tdt = {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32,
           np.dtype(np.int32): torch.int32, np.dtype(np.uint8): torch.uint8}[np.dtype(dtype)]
    return torch.empty(tuple(shape), dtype=tdt, pin_memory=True).numpy()  # view keeps it alive
