"""Host-buffer entry points through the raw C-ABI: an optional output left null changes none of
the outputs that are requested.  Each call is compared byte for byte with the call that requests
every output; all output arrays start from the same junk pattern, so an output that is not copied
back shows up too."""
import ctypes

import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from f1tenth_planning_b200.engine import Engine

pytestmark = pytest.mark.gpu


def _junk(a):
    a.view(np.uint8)[...] = 0x5A
    return a


def _vp(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _typed(a, t):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(t))


def _each_left_out(call, outs, optional):
    """call(bufs) once with every output, then once per optional output with that one left null
    (bufs[name] = None); the remaining outputs must come back byte-identical"""
    full = {k: _junk(np.empty_like(v)) for k, v in outs.items()}
    assert call(full) == 0
    assert all(full[k].tobytes() != _junk(np.empty_like(v)).tobytes() for k, v in outs.items())
    for drop in optional:
        bufs = {k: (None if k == drop else _junk(np.empty_like(v))) for k, v in outs.items()}
        assert call(bufs) == 0, drop
        for k, v in bufs.items():
            if v is not None:
                assert v.tobytes() == full[k].tobytes(), (drop, k)


def test_null_optional_outputs(ellipse, corridor):
    eng = Engine(kappa_max=3.0)
    eng.set_track(ellipse)
    eng.set_goal_grid(*synth.goal_grid(1))
    occ, origin, res = corridor
    eng.set_grid(occ, origin, res)
    L, h = eng._L, eng._h
    M, C = eng.n_samples, eng.n_candidates

    # f1l_plan_batch_prev over three pipeline chunks, previous paths updated in place (they are
    # outputs too: every call starts from the same paths)
    S, K = 3000, 2
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, K, 1009)
    P0 = np.ascontiguousarray(eng.plan_batch(poses, opp, n_opp).best_traj[:, :, 2])
    V0 = np.ones(S, np.uint8)
    V0[::3] = 0
    batch = dict(best_idx=np.zeros(S, np.int32), best_cost=np.zeros(S, np.float32),
                 best_traj=np.zeros((S, M, 4), np.float32), costs=np.zeros((S, C), np.float32),
                 flags=np.zeros((S, C), np.uint8), steer_speed=np.zeros((S, 2)),
                 prev_theta=P0, has_prev=V0)

    def plan(b):
        b["prev_theta"][...] = P0
        b["has_prev"][...] = V0
        return L.f1l_plan_batch_prev(h, _vp(poses), _vp(opp), _vp(n_opp), S, K, _vp(b["prev_theta"]),
                                     _vp(b["has_prev"]), 1, _vp(b["best_idx"]), _vp(b["best_cost"]),
                                     _vp(b["best_traj"]), _vp(b["costs"]), _vp(b["flags"]),
                                     _vp(b["steer_speed"]))
    _each_left_out(plan, batch, ["best_idx", "best_cost", "best_traj", "costs", "flags", "steer_speed"])

    B = 700
    rng = np.random.default_rng(1010)
    idx = rng.integers(0, ellipse.shape[0], B)
    states = np.ascontiguousarray(np.stack([ellipse[idx, 0] + rng.normal(0, 0.5, B),
                                            ellipse[idx, 1] + rng.normal(0, 0.5, B),
                                            ellipse[idx, 3] + rng.normal(0, 0.2, B),
                                            rng.uniform(1.0, 8.0, B)], axis=1))
    pp = dict(nearest=np.zeros((B, 4)), nearest_i=np.zeros(B, np.int32), lookahead=np.zeros((B, 4)),
              lookahead_i=np.zeros(B, np.int32), actuation=np.zeros((B, 2)), status=np.zeros(B, np.int32))
    poses3 = np.ascontiguousarray(states[:, :3])
    _each_left_out(lambda b: L.f1l_pure_pursuit_batch(h, _vp(poses3), B, 0.8, *(_vp(b[k]) for k in pp)),
                   pp, list(pp))

    fa = dict(front=np.zeros((B, 6)), nearest_i=np.zeros(B, np.int32))
    _each_left_out(lambda b: L.f1l_front_axle_batch(h, _vp(states), B, 0.33, 5.0, _vp(b["front"]),
                                                    _vp(b["nearest_i"])),
                   fa, ["nearest_i"])

    G = 300
    goals = np.ascontiguousarray(np.stack([rng.uniform(0.5, 3.5, G), rng.uniform(-1.0, 1.0, G),
                                           rng.uniform(-0.6, 0.6, G)], axis=1))
    gen = dict(states=np.zeros((G, M, 4), np.float32), params=np.zeros((G, 4), np.float32),
               flags=np.zeros(G, np.uint8))
    _each_left_out(lambda b: L.f1l_generate(h, _typed(goals, ctypes.c_double), G,
                                            _typed(b["states"], ctypes.c_float),
                                            _typed(b["params"], ctypes.c_float),
                                            _typed(b["flags"], ctypes.c_uint8)),
                   gen, ["params", "flags"])
