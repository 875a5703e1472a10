"""Closed-loop rollouts on the device (f1l_rollout_dev / Fleet.run).

Every comparison is teacher-forced, step by step from the traced states: device trig differs from
glibc's by an ulp, and one flipped argmin would separate two free-running rollouts for good."""
import ctypes
import math

import numpy as np
import pytest

from f1tenth_planning_b200 import _lib, synth
from f1tenth_planning_b200.rollout import CAR_HIT_MAP, CAR_HIT_CAR, CAR_NO_FEASIBLE
from oracle import c_oracle as co
from tests import helpers as H
from tests.test_gpu_batch_prev import _spielberg

pytestmark = pytest.mark.gpu

HIT = CAR_HIT_MAP | CAR_HIT_CAR
EPS = 1e-9   # pairs this close to touching / probes this close to a cell edge are exempt


def _ellipse_engine(ellipse, corridor, **cfg):
    la, wd = synth.goal_grid(4)
    eng, _, _ = H.make_pair(ellipse, la, wd, grid=corridor, kappa_max=3.0, **cfg)
    return eng, ellipse, corridor


def _spielberg_engine(golden_spielberg, **cfg):
    from f1tenth_planning_b200.engine import Engine
    wp, grid = _spielberg(golden_spielberg)
    eng = Engine(**cfg)
    eng.set_track(wp)
    eng.set_grid(*grid)
    eng.set_goal_grid(np.linspace(0.8, 3.0, 8), np.linspace(-0.6, 0.6, 9))
    return eng, wp, grid


def _race_poses(wp, S, G, spacing, seed, v=5.0, lat=0.25):
    """races spread over the raceline, the cars of a race `spacing` waypoints apart"""
    rng = np.random.default_rng(seed)
    n = wp.shape[0]
    base = np.repeat(np.linspace(0, n, S // G, endpoint=False).astype(int), G)
    idx = (base + spacing * np.tile(np.arange(G), S // G)) % n
    off = rng.normal(0.0, lat, S)
    psi = wp[idx, 3]
    return np.stack([wp[idx, 0] - off * np.sin(psi), wp[idx, 1] + off * np.cos(psi),
                     psi + rng.normal(0.0, 0.05, S), np.full(S, v)], axis=1)


def _race_opp(X, G):
    """[S,G-1,3] the other cars of each car's race in race order"""
    S = X.shape[0]
    R = X[:, :3].reshape(S // G, G, 3)
    out = np.zeros((S, max(G - 1, 1), 3))
    for j in range(G):
        out[j::G, :G - 1] = np.delete(R, j, axis=1)
    return out


# ---- float64 mirrors of the collision predicates ----------------------------------------------
def _map_hits(eng, grid, X, mode):
    """(hit [S], exempt [S]) of the footprint at X against the grid"""
    occ, (ox, oy), res = grid
    cfg = eng.config
    hl, hw = 0.5 * cfg.car_length, 0.5 * cfg.car_width
    c, s = np.cos(X[:, 2]), np.sin(X[:, 2])
    H_, W_ = occ.shape
    hit = np.zeros(X.shape[0], bool)
    ex = np.zeros(X.shape[0], bool)
    if mode == 1:
        edt = eng.get_edt(occ.shape).astype(np.int64)
        L, Wd = cfg.car_length, cfg.car_width
        t = math.sqrt(L * L / 36.0 + Wd * Wd / 4.0) / res + 1.4142135623730951
        t2 = int(math.floor(t * t)) + 1
        pts = [(k * (L / 3.0) * c, k * (L / 3.0) * s) for k in (-1, 0, 1)]
        pts = [(X[:, 0] + dx, X[:, 1] + dy) for dx, dy in pts]
    else:
        lx, ly, wx, wy = hl * c, hl * s, -(hw * s), hw * c
        pts = [((X[:, 0] + sa * lx) + sb * wx, (X[:, 1] + sa * ly) + sb * wy)
               for sa in (-1.0, 0.0, 1.0) for sb in (-1.0, 0.0, 1.0)]
    for px, py in pts:
        cx, cy = (px - ox) / res, (py - oy) / res
        col, row = np.floor(cx).astype(np.int64), np.floor(cy).astype(np.int64)
        ex |= (np.abs(cx - np.round(cx)) < EPS) | (np.abs(cy - np.round(cy)) < EPS)
        oob = (col < 0) | (col >= W_) | (row < 0) | (row >= H_)
        cc, rr = np.clip(col, 0, W_ - 1), np.clip(row, 0, H_ - 1)
        hit |= oob | ((edt[rr, cc] < t2) if mode == 1 else (occ[rr, cc] != 0))
    return hit, ex


def _car_hits(eng, X, G):
    cfg = eng.config
    hl, hw = 0.5 * cfg.car_length, 0.5 * cfg.car_width
    S = X.shape[0]
    hit = np.zeros(S, bool)
    ex = np.zeros(S, bool)
    c, s = np.cos(X[:, 2]), np.sin(X[:, 2])
    for i in range(S):
        for j in range(i - i % G, i - i % G + G):
            if j == i:
                continue
            tx, ty = X[j, 0] - X[i, 0], X[j, 1] - X[i, 1]
            cc = abs(c[i] * c[j] + s[i] * s[j])
            ss = abs(s[i] * c[j] - c[i] * s[j])
            rl, rw = hl + (hl * cc + hw * ss), hw + (hl * ss + hw * cc)
            e = (abs(tx * c[i] + ty * s[i]), abs(ty * c[i] - tx * s[i]),
                 abs(tx * c[j] + ty * s[j]), abs(ty * c[j] - tx * s[j]))
            m = min(rl - e[0], rw - e[1], rl - e[2], rw - e[3])
            hit[i] |= m > 0
            ex[i] |= abs(m) < EPS
    return hit, ex


def _step_ref(eng, grid, X, ss, feasible, status, G, substeps, mode, dt=0.01, max_steer=0.4189,
              max_accel=9.51, v_max=math.inf):
    """the stated model for one planning step -> (state, status, exempt)"""
    X = X.copy()
    st = status & np.uint8(0xFF ^ CAR_NO_FEASIBLE)
    st[~feasible] |= CAR_NO_FEASIBLE
    steer = np.clip(ss[:, 0], -max_steer, max_steer)
    target = np.where(feasible, np.minimum(ss[:, 1], v_max), 0.0)
    tan_s = np.tan(steer)
    wb = eng.config.wheelbase
    ex = np.zeros(X.shape[0], bool)
    for _ in range(substeps):
        frozen = (st & HIT) != 0
        v = X[:, 3] + np.clip(target - X[:, 3], -(max_accel * dt), max_accel * dt)
        nx = np.stack([X[:, 0] + v * np.cos(X[:, 2]) * dt, X[:, 1] + v * np.sin(X[:, 2]) * dt,
                       X[:, 2] + v / wb * tan_s * dt, v], axis=1)
        X = np.where(frozen[:, None], X, nx)
        X[frozen, 3] = 0.0
        hm, e1 = _map_hits(eng, grid, X, mode)
        hc, e2 = _car_hits(eng, X, G)
        ex |= e1 | e2
        st = st | np.where(hm, CAR_HIT_MAP, 0).astype(np.uint8) | np.where(hc, CAR_HIT_CAR, 0).astype(np.uint8)
        X[(st & HIT) != 0, 3] = 0.0
    return X, st.astype(np.uint8), ex


def _np(tr):
    return type(tr)(*(t.cpu().numpy() for t in tr))


def _teacher_forced(eng, grid, tr, final, G, substeps, mode, P0=None, V0=None, v_max=math.inf):
    """every step of a traced run against plan_batch + the numpy model; returns (exempt, hits)"""
    T, S = tr.best_idx.shape
    P = np.zeros((S, eng.n_samples), np.float32) if P0 is None else P0.copy()
    V = np.zeros(S, np.uint8) if V0 is None else V0.copy()
    st = np.zeros(S, np.uint8)
    n_ex = 0
    for k in range(T):
        X = tr.state[k]
        if G > 1:
            b = eng.plan_batch(X, _race_opp(X, G), np.full(S, G - 1, np.int32), want_traj=False,
                               want_costs=False, prev_theta=P, has_prev=V, update_prev=True)
        else:
            b = eng.plan_batch(X, want_traj=False, want_costs=False, prev_theta=P, has_prev=V,
                               update_prev=True)
        assert np.array_equal(b.best_idx, tr.best_idx[k]), k
        assert np.array_equal(b.steer_speed, tr.steer_speed[k]), k
        Xn, stn, ex = _step_ref(eng, grid, X, tr.steer_speed[k], np.isfinite(b.best_cost), st, G,
                                substeps, mode, v_max=v_max)
        nxt = tr.state[k + 1] if k + 1 < T else final
        ok = ~ex
        n_ex += int(ex.sum())
        assert np.abs(Xn[ok] - nxt[ok]).max(initial=0.0) <= 1e-10, k
        assert np.array_equal(stn[ok], tr.status[k][ok]), (k, np.nonzero(stn != tr.status[k]))
        st = tr.status[k]
    return n_ex, int(((tr.status[-1] & HIT) != 0).sum())


@pytest.mark.parametrize("G,substeps", [(1, 1), (1, 5), (4, 1), (4, 5)])
def test_steps_equal_batch_planning(ellipse, corridor, G, substeps):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S = 32
    X0 = _race_poses(wp, S, G, 4, 2001 + G, lat=0.4)
    fleet = eng.fleet(X0, group=G)
    tr = _np(fleet.run(60, substeps=substeps, v_max=6.0, trace=True))
    assert np.array_equal(tr.state[0], X0)
    n_ex, hits = _teacher_forced(eng, grid, tr, fleet.state.cpu().numpy(), G, substeps, 0, v_max=6.0)
    assert n_ex <= 2, n_ex
    moved = np.hypot(*(fleet.state.cpu().numpy()[:, :2] - X0[:, :2]).T)
    assert (moved[(tr.status[-1] & HIT) == 0] > 0.5).all()


def test_steps_equal_batch_planning_spielberg(golden_spielberg):
    eng, wp, grid = _spielberg_engine(golden_spielberg)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 6, 2011)
    fleet = eng.fleet(X0, group=G)
    tr = _np(fleet.run(60, substeps=5, v_max=5.0, trace=True))
    n_ex, _ = _teacher_forced(eng, grid, tr, fleet.state.cpu().numpy(), G, 5, 0, v_max=5.0)
    assert n_ex <= 2, n_ex


@pytest.mark.parametrize("mode", [0, 1])
def test_crafted_collisions(ellipse, corridor, mode):
    eng, wp, grid = _ellipse_engine(ellipse, corridor, collision_mode=mode)
    # poses on the raceline, k waypoints (about 0.19 m each) after waypoint 100
    pose = lambda k, v=3.0: [wp[100 + k, 0], wp[100 + k, 1], wp[100 + k, 3], v]   # noqa: E731
    X0 = np.array([
        pose(0), pose(1),                  # race 0: overlapping
        [0.0, 0.0, 0.0, 3.0], pose(30),    # race 1: the first car inside the wall (the oval's centre)
        pose(60), pose(90),                # race 2
        pose(120), pose(150),              # races 3 and 4: cars 7 and 8 at identical poses
        pose(150), pose(180),
    ])
    fleet = eng.fleet(X0, group=2)
    tr = _np(fleet.run(8, substeps=2, trace=True))
    st = tr.status
    assert (st[0, :2] & CAR_HIT_CAR).all() and (st[:, :2] & CAR_HIT_CAR).all()
    assert (st[0, 2] & CAR_HIT_MAP) and not (st[0, 3] & HIT)
    assert not (st[:, 3:7] & HIT).any()
    assert not (st[:, 7:9] & CAR_HIT_CAR).any()   # identical poses, different races
    # frozen: pose of the first hit kept, v = 0 from then on
    for c in (0, 1, 2):
        assert (tr.state[1:, c, 3] == 0).all()
        assert (tr.state[1:, c, :3] == tr.state[1, c, :3]).all()
    # a frozen car is still an opponent: car 3 plans around frozen car 2 0.8 m ahead of it
    X1 = np.array([pose(0), pose(100), pose(214, 0.0), pose(210)])
    f2 = eng.fleet(X1, group=2)
    f2.status[2] = CAR_HIT_MAP
    tr2 = _np(f2.run(10, trace=True))
    assert (tr2.state[:, 2, :3] == X1[2, :3]).all() and (tr2.state[1:, 2, 3] == 0).all()
    P, V = np.zeros((4, eng.n_samples), np.float32), np.zeros(4, np.uint8)
    Pn, Vn = P.copy(), V.copy()
    differs = 0
    for k in range(10):
        X = tr2.state[k]
        b = eng.plan_batch(X, _race_opp(X, 2), np.ones(4, np.int32), want_traj=False, want_costs=False,
                           prev_theta=P, has_prev=V, update_prev=True)
        assert np.array_equal(b.best_idx, tr2.best_idx[k]), k
        alone = eng.plan_batch(X, want_traj=False, want_costs=False, prev_theta=Pn, has_prev=Vn,
                               update_prev=False)
        differs += int(alone.best_idx[3] != b.best_idx[3])
        Pn[:], Vn[:] = P, V
    assert differs > 0


def _seg_s(wp):
    d = np.diff(wp[:, :2], axis=0)
    ln = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
    cum = np.concatenate([[0.0], np.cumsum(ln)])
    g = wp[0, :2] - wp[-1, :2]
    return cum, ln, cum[-1] + math.sqrt(g[0] * g[0] + g[1] * g[1])


def _wrap(ds, lap):
    ds = np.where(ds >= 0.5 * lap, ds - lap, ds)
    return np.where(ds < -0.5 * lap, ds + lap, ds)


def test_progress_tracking(ellipse, corridor):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    n = wp.shape[0]
    cum, ln, lap = _seg_s(wp)
    S = 16
    X0 = _race_poses(wp, S, 1, 0, 2021, v=5.0, lat=0.3)
    X0[0] = [wp[n - 30, 0], wp[n - 30, 1], wp[n - 30, 3], 5.0]   # 30 waypoints before the seam
    fleet = eng.fleet(X0, group=1)
    prev_s, prev_p = None, np.zeros(S)
    seam = []
    checked = 0
    for k in range(40):
        if k == 20:
            fleet.track_i[3] = -1   # re-acquire: progress stays as given
        fleet.run(1, substeps=5)
        X = fleet.state.cpu().numpy()
        ti, ts = fleet.track_i.cpu().numpy(), fleet.track_s.cpu().numpy()
        prog = fleet.progress.cpu().numpy()
        for c in range(S):
            _, dist, t, i = co.nearest_point(X[c, :2], wp[:, :2])
            if dist < 1.0 and 0.0 < t < 1.0 and not (fleet.status[c].item() & HIT):
                assert ti[c] == i, (k, c)
                assert abs((ts[c] - cum[i]) / ln[i] - t) < 2e-12, (k, c)
                checked += 1
        s = ts
        if prev_s is not None:
            inc = _wrap(s - prev_s, lap)
            assert np.abs((prog - prev_p) - inc).max() <= 1e-9, k
        prev_s, prev_p = s, prog
        seam.append(ti[0])
    assert checked > 400
    assert max(seam) > n - 20 and min(seam) < 20   # car 0 crossed the seam ...
    d = np.hypot(*(fleet.state.cpu().numpy()[0, :2] - X0[0, :2]))
    assert 0.9 * d < prog[0] < 1.2 * d + 1.0   # ... and kept counting


def test_continuity_and_reset(ellipse, corridor):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 5, 2031)
    a, b = eng.fleet(X0, group=G), eng.fleet(X0, group=G)
    a.run(30, substeps=2)
    a.run(30, substeps=2)
    b.run(60, substeps=2)
    for name in ("state", "prev_theta", "has_prev", "status", "progress", "track_i", "track_s"):
        assert np.array_equal(getattr(a, name).cpu().numpy(), getattr(b, name).cpu().numpy()), name
    # reset mid-run (G = 1): the reset cars agree with a fresh fleet of the same size
    c = eng.fleet(X0, group=1)
    c.run(20)
    cars = [3, 17]
    newp = X0[[10, 25]] + np.array([0.1, 0.05, 0.0, 0.0])
    c.reset(cars, newp)
    fresh = eng.fleet(c.state, group=1)
    tc, tf = _np(c.run(15, trace=True)), _np(fresh.run(15, trace=True))
    for f in tc._fields:
        assert np.array_equal(getattr(tc, f)[:, cars], getattr(tf, f)[:, cars]), f
    assert np.array_equal(c.progress.cpu().numpy()[cars], fresh.progress.cpu().numpy()[cars])


def test_scale(ellipse, corridor):
    import torch
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 100000, 4
    X0, _ = synth.random_poses(wp, S, np.random.default_rng(2041))
    fleet = eng.fleet(X0, group=G)
    tr = fleet.run(3, substeps=2, trace=True)
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
    for t in (tr.state, tr.steer_speed, tr.progress, fleet.state, fleet.progress):
        assert torch.isfinite(t).all()


def test_bad_arguments_are_rejected(ellipse, corridor):
    import torch
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    X0 = _race_poses(wp, 8, 4, 5, 2051)
    for bad in (dict(group=0), dict(group=18), dict(group=3)):
        with pytest.raises(ValueError):
            eng.fleet(X0, **bad)
    for bad in (np.zeros((8, 3)), np.zeros(8), np.zeros((0, 4))):
        with pytest.raises(ValueError):
            eng.fleet(bad)
    fleet = eng.fleet(X0, group=4)
    for kw in (dict(n_steps=-1), dict(substeps=0), dict(dt=0.0), dict(dt=-0.01), dict(dt=math.nan),
               dict(max_steer=0.0), dict(max_accel=math.nan), dict(v_max=0.0), dict(v_max=math.nan)):
        args = dict(n_steps=1)
        args.update(kw)
        with pytest.raises(ValueError):
            fleet.run(**args)
    good = fleet.state
    for bad in (good.float(), good.cpu(), good.t().contiguous().t()[:, :4], torch.zeros(4, 4, dtype=torch.float64,
                                                                                          device=good.device)):
        fleet.state = bad
        with pytest.raises(ValueError):
            fleet.run(1)
    fleet.state = good
    assert fleet.run(0) is None
    # the raw ABI
    L = eng._L
    fl = fleet._buffers()
    S = fleet.n_cars

    def call(rc=None, fl_=fl, S_=S, T=1, h=eng._h):
        if rc is None:
            rc = _lib.RolloutConfig(0.01, 1, 4, 0.4189, 9.51, math.inf)
        return L.f1l_rollout_dev(h, ctypes.byref(rc) if rc is not False else None,
                                 ctypes.byref(fl_) if fl_ is not None else None, S_, T, None, None)

    ok = dict(dt=0.01, substeps=1, group=4, max_steer=0.4189, max_accel=9.51, v_max=math.inf)
    for kw in (dict(group=0), dict(group=18), dict(group=3), dict(substeps=0), dict(dt=0.0),
               dict(dt=math.nan), dict(max_steer=-1.0), dict(max_accel=0.0), dict(v_max=math.nan)):
        cfg = dict(ok)
        cfg.update(kw)
        assert call(_lib.RolloutConfig(**cfg)) == -1, kw
    assert call(T=-1) == -1
    assert call(h=None) == -1
    assert call(rc=False) == -1
    assert call(fl_=None) == -1
    assert call(fl_=_lib.FleetBuffers(fl.state, fl.prev_theta, None, fl.status, fl.progress, fl.track_i,
                                      fl.track_s)) == -1
    assert call(S_=6) == -1 and call(S_=0) == -1
    before = fleet.state.clone()
    assert call(T=0) == 0
    torch.cuda.synchronize()
    assert torch.equal(before, fleet.state)
