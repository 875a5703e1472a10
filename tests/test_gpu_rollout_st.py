"""Closed-loop rollouts of single-track cars on the device (f1l_rollout_st_dev, Fleet with a vehicle).

As in test_gpu_rollout.py every comparison is teacher-forced: each traced step is planned again by
plan_batch and stepped by the numpy restatement of tests/st_model.py from the traced state and
dyn, so device trig that differs from glibc's by an ulp cannot separate two rollouts."""
import ctypes
import math

import numpy as np
import pytest

from f1tenth_planning_b200 import _lib, synth
from f1tenth_planning_b200.rollout import CAR_HIT_MAP, CAR_HIT_CAR, CAR_NO_FEASIBLE, SingleTrackTrace, Vehicle
from tests import st_model as stm
from tests.test_gpu_rollout import (_car_hits, _ellipse_engine, _map_hits, _np, _race_opp, _race_poses,
                                    _spielberg_engine)

pytestmark = pytest.mark.gpu

HIT = CAR_HIT_MAP | CAR_HIT_CAR


def _st_step_ref(eng, grid, X, D, ss, feasible, status, G, substeps, mode, v_max, dt=0.01, max_steer=0.4189,
                 max_accel=9.51):
    """the stated single-track model for one planning step -> (state, dyn, status, exempt)"""
    X, D = X.copy(), D.copy()
    st = status & np.uint8(0xFF ^ CAR_NO_FEASIBLE)
    st[~feasible] |= CAR_NO_FEASIBLE
    steer = np.clip(ss[:, 0], -max_steer, max_steer)
    target = np.where(feasible, np.minimum(ss[:, 1], v_max), 0.0)
    ex = np.zeros(X.shape[0], bool)
    for _ in range(substeps):
        frozen = (st & HIT) != 0
        Xn, Dn = stm.substep(X, D, steer, target, dt, max_accel)
        X = np.where(frozen[:, None], X, Xn)
        D = np.where(frozen[:, None], D, Dn)
        X[frozen, 3] = 0.0
        D[frozen, 1:] = 0.0
        hm, e1 = _map_hits(eng, grid, X, mode)
        hc, e2 = _car_hits(eng, X, G)
        ex |= e1 | e2
        st = st | np.where(hm, CAR_HIT_MAP, 0).astype(np.uint8) | np.where(hc, CAR_HIT_CAR, 0).astype(np.uint8)
        hit = (st & HIT) != 0
        X[hit, 3] = 0.0
        D[hit, 1:] = 0.0
    return X, D, st.astype(np.uint8), ex


def _teacher_forced(eng, grid, tr, final, final_dyn, G, substeps, v_max, weights=None):
    """every traced step against plan_batch + the numpy model; v_max per step; returns the number
    of exempt (near-touching) cars"""
    T, S = tr.best_idx.shape
    v_max = np.broadcast_to(np.asarray(v_max, np.float64), (T,))
    P = np.zeros((S, eng.n_samples), np.float32)
    V = np.zeros(S, np.uint8)
    st = np.zeros(S, np.uint8)
    n_ex = 0
    for k in range(T):
        X, D = tr.state[k], tr.dyn[k]
        opp = dict(opponents=_race_opp(X, G), n_opp=np.full(S, G - 1, np.int32)) if G > 1 else {}
        b = eng.plan_batch(X, **opp, want_traj=False, want_costs=False, prev_theta=P, has_prev=V,
                           update_prev=True, weights=weights)
        assert np.array_equal(b.best_idx, tr.best_idx[k]), k
        assert np.array_equal(b.steer_speed, tr.steer_speed[k]), k
        Xn, Dn, stn, ex = _st_step_ref(eng, grid, X, D, tr.steer_speed[k], np.isfinite(b.best_cost), st, G,
                                       substeps, 0, v_max[k])
        nxt = tr.state[k + 1] if k + 1 < T else final
        nd = tr.dyn[k + 1] if k + 1 < T else final_dyn
        ok = ~ex
        n_ex += int(ex.sum())
        assert np.abs(Xn[ok] - nxt[ok]).max(initial=0.0) <= 1e-10, k
        assert np.abs(Dn[ok] - nd[ok]).max(initial=0.0) <= 1e-10, k
        assert np.array_equal(stn[ok], tr.status[k][ok]), (k, np.nonzero(stn != tr.status[k]))
        st = tr.status[k]
    return n_ex


def _final(fleet):
    return fleet.state.cpu().numpy(), fleet.dyn.cpu().numpy()


@pytest.mark.parametrize("G,substeps", [(1, 1), (1, 5), (4, 1), (4, 5)])
def test_steps_equal_batch_planning_and_the_model(ellipse, corridor, G, substeps):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S = 32
    X0 = _race_poses(wp, S, G, 4, 3001 + G, lat=0.4)
    fleet = eng.fleet(X0, group=G, vehicle=Vehicle())
    tr = _np(fleet.run(60, substeps=substeps, v_max=6.0, trace=True))
    assert type(tr) is SingleTrackTrace and tr.dyn.shape == (60, S, 3)
    assert np.array_equal(tr.state[0], X0) and not tr.dyn[0].any()
    assert _teacher_forced(eng, grid, tr, *_final(fleet), G, substeps, 6.0) <= 2
    X = fleet.state.cpu().numpy()
    moved = np.hypot(*(X[:, :2] - X0[:, :2]).T)
    live = (tr.status[-1] & HIT) == 0
    assert (moved[live] > 0.5).all()
    assert (np.abs(tr.dyn[1:, :, 2]) > 1e-3).any()   # the cars slip


def test_steps_equal_batch_planning_spielberg(golden_spielberg):
    eng, wp, grid = _spielberg_engine(golden_spielberg)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 6, 3011)
    fleet = eng.fleet(X0, group=G, vehicle=Vehicle())
    tr = _np(fleet.run(60, substeps=5, v_max=5.0, trace=True))
    assert _teacher_forced(eng, grid, tr, *_final(fleet), G, 5, 5.0) <= 2


def test_crossing_v_kin_both_ways(ellipse, corridor):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 16, 4
    X0 = _race_poses(wp, S, G, 6, 3021, v=0.0, lat=0.2)
    fleet = eng.fleet(X0, group=G, vehicle=Vehicle())
    a = _np(fleet.run(40, substeps=2, v_max=6.0, trace=True))
    b = _np(fleet.run(60, substeps=2, v_max=0.2, trace=True))
    tr = SingleTrackTrace(*(np.concatenate([x, y]) for x, y in zip(a, b)))
    v = np.concatenate([tr.state[:, :, 3], fleet.state.cpu().numpy()[None, :, 3]])
    v_kin = Vehicle().v_kin
    crossed = (v[:41] > v_kin).any(0) & (v[-1] < v_kin) & ((tr.status[-1] & HIT) == 0)
    assert (v[0] == 0).all() and crossed.sum() >= S // 2, (v[40], v[-1], tr.status[-1])
    assert _teacher_forced(eng, grid, tr, *_final(fleet), G, 2, [6.0] * 40 + [0.2] * 60) <= 2


def test_continuity_and_reset(ellipse, corridor):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 5, 3031)
    a, b = eng.fleet(X0, group=G, vehicle=Vehicle()), eng.fleet(X0, group=G, vehicle=Vehicle())
    a.run(30, substeps=2)
    a.run(30, substeps=2)
    b.run(60, substeps=2)
    for name in ("state", "dyn", "prev_theta", "has_prev", "status", "progress", "track_i", "track_s"):
        assert np.array_equal(getattr(a, name).cpu().numpy(), getattr(b, name).cpu().numpy()), name
    assert a.dyn.abs().max().item() > 0
    c = eng.fleet(X0, group=1, vehicle=Vehicle())
    c.run(20)
    cars = [3, 17]
    c.reset(cars, X0[[10, 25]] + np.array([0.1, 0.05, 0.0, 0.0]))
    assert not c.dyn[cars].any() and c.dyn.abs().max().item() > 0
    fresh = eng.fleet(c.state, group=1, vehicle=Vehicle())
    tc, tf = _np(c.run(15, trace=True)), _np(fresh.run(15, trace=True))
    for f in tc._fields:
        assert np.array_equal(getattr(tc, f)[:, cars], getattr(tf, f)[:, cars]), f
    assert np.array_equal(c.dyn.cpu().numpy()[cars], fresh.dyn.cpu().numpy()[cars])


def test_per_car_weights(ellipse, corridor):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 4, 3041)
    W = np.random.default_rng(3041).uniform(0.0, 2.0, (S, _lib.N_TERMS)).astype(np.float32)
    fleet = eng.fleet(X0, group=G, weights=W, vehicle=Vehicle())
    tr = _np(fleet.run(1, substeps=2, v_max=6.0, trace=True))
    assert _teacher_forced(eng, grid, tr, *_final(fleet), G, 2, 6.0, weights=W) <= 2
    plain = eng.plan_batch(X0, _race_opp(X0, G), np.full(S, G - 1, np.int32), want_traj=False, want_costs=False)
    assert not np.array_equal(plain.best_idx, tr.best_idx[0])


def test_scale(ellipse, corridor):
    import torch
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 100000, 4
    X0, _ = synth.random_poses(wp, S, np.random.default_rng(3051))
    fleet = eng.fleet(X0, group=G, vehicle=Vehicle())
    tr = fleet.run(1, substeps=2, trace=True)
    fleet.run(19, substeps=2)
    dev = fleet.state.device
    opp = torch.zeros(S, 16, 3, dtype=torch.float64, device=dev)
    opp[:, :G - 1] = torch.from_numpy(_race_opp(X0, G)).to(dev)
    idx = torch.empty(S, dtype=torch.int32, device=dev)
    ss = torch.empty(S, 2, dtype=torch.float64, device=dev)
    P = torch.zeros(S, eng.n_samples, dtype=torch.float32, device=dev)
    V = torch.zeros(S, dtype=torch.uint8, device=dev)
    eng.plan_batch_dev(torch.from_numpy(X0).to(dev), opp, torch.full((S,), G - 1, dtype=torch.int32, device=dev),
                       best_idx=idx, steer_speed=ss, prev_theta=P, has_prev=V, update_prev=True)
    torch.cuda.synchronize(dev)
    assert torch.equal(idx, tr.best_idx[0]) and torch.equal(ss, tr.steer_speed[0])
    for t in (tr.state, tr.dyn, fleet.state, fleet.dyn, fleet.progress):
        assert torch.isfinite(t).all()
    assert fleet.dyn.abs().max().item() > 0


def test_bad_arguments_are_rejected(ellipse, corridor):
    import torch
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    X0 = _race_poses(wp, 8, 4, 5, 3061)
    for f in Vehicle._fields:
        for val in ([-1.0, math.nan] if f == "h" else [0.0, -1.0, math.nan]):
            with pytest.raises(ValueError):
                eng.fleet(X0, group=4, vehicle=Vehicle(**{f: val}))
    fleet = eng.fleet(X0, group=4, vehicle=Vehicle())
    good = fleet.dyn
    for bad in (good.float(), good.cpu(), torch.zeros(8, 4, dtype=torch.float64, device=good.device)[:, :3],
                torch.zeros(4, 3, dtype=torch.float64, device=good.device),
                torch.zeros(8, 2, dtype=torch.float64, device=good.device)):
        fleet.dyn = bad
        with pytest.raises(ValueError):
            fleet.run(1)
    fleet.dyn = good
    fleet.vehicle = Vehicle(v_kin=0.0)
    with pytest.raises(ValueError):
        fleet.run(1)
    fleet.vehicle = Vehicle()
    assert fleet.run(0) is None
    # the raw ABI
    L = eng._L
    fl = fleet._buffers()
    rc = _lib.RolloutConfig(0.01, 1, 4, 0.4189, 9.51, math.inf)
    dyn = ctypes.c_void_p(good.data_ptr())

    def call(veh, dyn_=dyn, rc_=rc, T=1):
        return L.f1l_rollout_st_dev(eng._h, ctypes.byref(rc_), ctypes.byref(veh) if veh is not None else None,
                                    ctypes.byref(fl), dyn_, None, 8, T, None, None, None)

    ok = _lib.Vehicle()
    assert L.f1l_default_vehicle(ctypes.byref(ok)) == 0
    for f, _ in _lib.Vehicle._fields_:
        for val in ([-1.0, math.nan] if f == "h" else [0.0, math.nan]):
            v = _lib.Vehicle.from_buffer_copy(ok)
            setattr(v, f, val)
            assert call(v) == -1, (f, val)
    assert call(None) == -1
    assert call(ok, dyn_=None) == -1
    assert call(ok, rc_=_lib.RolloutConfig(0.01, 1, 3, 0.4189, 9.51, math.inf)) == -1
    before = (fleet.state.clone(), fleet.dyn.clone())
    assert call(ok, T=0) == 0
    zero_h = _lib.Vehicle.from_buffer_copy(ok)
    zero_h.h = 0.0
    assert call(zero_h, T=0) == 0
    torch.cuda.synchronize()
    assert torch.equal(before[0], fleet.state) and torch.equal(before[1], fleet.dyn)
