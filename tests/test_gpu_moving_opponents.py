"""Moving opponents on the device (f1l_plan_motion, f1l_plan_batch_motion*, f1l_rollout_predict_dev):
zero velocities change nothing, the kernel's flags equal the float32 mirror on its own trajectories,
the answers agree with the float64 oracle outside the margin classes, the single-query graph keeps
static and moving calls apart, and a predicting fleet plans exactly as the batch call does."""
import ctypes
import math

import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from f1tenth_planning_b200.rollout import Vehicle
from oracle import c_oracle as co
from tests import motion_oracle as MO
from tests import helpers as H
from tests.test_gpu_batch_prev import NUDGE, _paths
from tests.test_gpu_rollout import _np, _race_opp, _race_poses

pytestmark = pytest.mark.gpu

SINGLE_M = [2, 32, 33, 64, 100, 104, 105, 128, 129, 200, 256]


def _shape11(eng):
    out = (ctypes.c_int32 * 11)()
    assert eng._L.f1l_last_eval_shape(eng._h, out, 11) == 0
    return list(out)


def _pair(track, grid, grid_cfg=4, **cfg):
    la, wd = synth.goal_grid(grid_cfg)
    return H.make_pair(track, la, wd, grid=grid, kappa_max=3.0, **cfg)


def _assert_same_detail(a, b):
    for k in ("costs", "terms", "flags", "goals", "params", "best_traj", "best_traj_map", "states", "headings"):
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None) == (y is None), k
        if x is not None:
            assert np.array_equal(x, y, equal_nan=True), k
    for k in ("best_idx", "best_cost", "steer", "speed", "no_feasible", "tracker_found"):
        assert getattr(a, k) == getattr(b, k), k


# ---- 1. zero velocities are bit-identical ------------------------------------------------------
@pytest.mark.parametrize("M", SINGLE_M)
def test_zero_velocities_single_query(ellipse, corridor, M):
    eng, _, _ = _pair(ellipse, corridor, n_samples=M)
    for seed in (3, 8):
        pose, opp = H.scenario(ellipse, seed, 6)
        kw = dict(update_prev=False, want_states=True, want_headings=True, want_map=True)
        d = eng.plan(pose, opp, **kw)
        assert _shape11(eng)[10] == 0
        dm = eng.plan(pose, opp, opponent_velocities=np.zeros((6, 2)), **kw)
        assert _shape11(eng)[10] == 1
        _assert_same_detail(d, dm)


def test_zero_velocities_dense_single_query(ellipse, corridor):
    """the 256 x 256 grid: a lone dense query on the persistent grid, its MO twin"""
    eng, _, _ = _pair(ellipse, corridor, grid_cfg=5)
    pose, opp = H.scenario(ellipse, 11, 8)
    d = eng.plan(pose, opp, update_prev=False)
    shape = _shape11(eng)
    dm = eng.plan(pose, opp, update_prev=False, opponent_velocities=np.zeros((8, 2)))
    shape_m = _shape11(eng)
    assert shape[8] == 1 and shape[9:] == [0, 0]
    assert shape_m[:9] == shape[:9] and shape_m[9:] == [1, 1]
    _assert_same_detail(d, dm)


@pytest.mark.parametrize("M,S", [(100, 96), (100, 5000), (200, 96), (33, 96)])
def test_zero_velocities_batch(ellipse, corridor, M, S):
    eng, _, _ = _pair(ellipse, corridor, n_samples=M)
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 8, 1201)
    P, V = _paths(eng, poses, opp, n_opp)
    poses = poses + NUDGE
    zero = np.zeros((S, 8, 2))
    W = np.random.default_rng(2).uniform(0.0, 2.0, (S, 5)).astype(np.float32)
    for extra in (dict(), dict(weights=W), dict(prev_theta=P, has_prev=V), dict(weights=W, prev_theta=P, has_prev=V)):
        b = eng.plan_batch(poses, opp, n_opp, want_flags=True, want_terms=True, **extra)
        bm = eng.plan_batch(poses, opp, n_opp, want_flags=True, want_terms=True, opponent_velocities=zero, **extra)
        assert _shape11(eng)[10] == 1
        for k in b._fields:
            x, y = getattr(b, k), getattr(bm, k)
            if x is not None:
                assert np.array_equal(x, y, equal_nan=True), (k, sorted(extra))


def test_zero_velocities_batch_device_and_update_prev(ellipse, corridor):
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    S = 256
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 4, 1301)
    P, V = _paths(eng, poses, opp, n_opp)
    dev = torch.device("cuda", eng.device)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    outs = []
    for vel in (None, np.zeros((S, 4, 2))):
        idx = torch.empty(S, dtype=torch.int32, device=dev)
        costs = torch.empty(S, eng.n_candidates, dtype=torch.float32, device=dev)
        pt, vt = t(P), t(V)
        eng.plan_batch_dev(t(poses), t(opp), t(n_opp), best_idx=idx, costs=costs, prev_theta=pt, has_prev=vt,
                           update_prev=True, opponent_velocities=None if vel is None else t(vel))
        torch.cuda.synchronize(dev)
        outs.append([a.cpu().numpy() for a in (idx, costs, pt, vt)])
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


# ---- 2. teacher-forced flags -------------------------------------------------------------------
def _crafted(track, seed):
    """(pose, opp [K,3], vel [K,2]) around a random pose, the cases where prediction matters:
    head-on, crossing, an overtaker from behind, a faster leader, and fast opponents 6-15 m away"""
    rng = np.random.default_rng(seed)
    poses, _ = synth.random_poses(track, 1, rng)
    pose = poses[0]
    x, y, th, v = pose
    c, s = math.cos(th), math.sin(th)
    loc = lambda f, l: (x + c * f - s * l, y + s * f + c * l)
    opp, vel = [], []
    def add(f, l, h, speed):
        opp.append(loc(f, l) + (th + h,))
        vel.append((speed * math.cos(th + h), speed * math.sin(th + h)))
    add(rng.uniform(4.0, 7.0), rng.normal(0.0, 0.3), math.pi, rng.uniform(2.0, 5.0))          # head-on
    add(rng.uniform(1.5, 3.0), -rng.uniform(2.0, 4.0), math.pi / 2, rng.uniform(3.0, 6.0))    # crossing
    add(-rng.uniform(1.0, 2.0), rng.normal(0.0, 0.4), 0.0, v + rng.uniform(2.0, 5.0))         # overtaker
    add(rng.uniform(0.8, 1.5), rng.normal(0.0, 0.3), 0.0, v + rng.uniform(0.5, 3.0))          # faster leader
    for _ in range(3):                                                                       # far and fast
        a = rng.uniform(-0.6, 0.6)
        r = rng.uniform(6.0, 15.0)
        add(r * math.cos(a), r * math.sin(a), math.pi + a, rng.uniform(8.0, 15.0))
    return pose, np.array(opp), np.array(vel)


def test_teacher_forced_flags_bit_exact(ellipse):
    la, wd = synth.goal_grid(3)
    grid = synth.corridor_grid(half_width=1.0)
    eng, cfg, world = H.make_pair(ellipse, la, wd, grid=grid)
    hl, hw = np.float32(0.5 * cfg.car_length), np.float32(0.5 * cfg.car_width)
    rc2 = np.float32(4.0 * ((0.5 * cfg.car_length) ** 2 + (0.5 * cfg.car_width) ** 2))
    n_checked = n_opp_hits = n_changed = 0
    for seed in range(8):
        pose, opp, vel = _crafted(ellipse, 500 + seed)
        d = eng.plan(pose, opp, update_prev=False, want_states=True, want_headings=True, opponent_velocities=vel)
        f, i = eng.debug_query_ctx()
        k_t, wl = eng.debug_motion_ctx()
        ve = max(pose[3], 1.0)
        assert k_t == np.float32(1.0 / ((cfg.n_samples - 1) * ve))
        assert np.allclose(wl[:len(opp)], [[math.cos(pose[2]) * a + math.sin(pose[2]) * b,
                                            -math.sin(pose[2]) * a + math.cos(pose[2]) * b] for a, b in vel],
                           rtol=1e-6, atol=1e-5)
        assert not wl[len(opp):].any()
        mirror = MO.collide_f32_motion(d.states, d.headings, d.params, f[8:].reshape(16, 4), wl, k_t, int(i[5]),
                                       f[2:8], i[0:2], grid[0], hl, hw, rc2)
        valid = (d.flags & 1) != 0
        assert np.array_equal(mirror[valid], d.flags[valid] & 6), seed
        static = eng.plan(pose, opp, update_prev=False)
        n_changed += int(((static.flags ^ d.flags) & 2)[valid].astype(bool).sum())
        n_checked += int(valid.sum())
        n_opp_hits += int((d.flags[valid] & 2).astype(bool).sum())
    assert n_checked > 10000 and n_opp_hits > 500 and n_changed > 500


# ---- 3. parity with the float64 oracle -----------------------------------------------------------
def test_parity_with_oracle_and_batch_equals_single(ellipse, corridor):
    eng, cfg, world = _pair(ellipse, corridor)
    counts = {"argmin_mismatch": 0, "argmin:cost_gap<1e-5": 0}
    cases = [_crafted(ellipse, 900 + s) for s in range(12)]
    rng = np.random.default_rng(3)
    for s in range(12):
        pose, opp = H.scenario(ellipse, 700 + s, 6)
        cases.append((pose, opp, synth.opponent_velocities(ellipse, opp, rng)))
    for pose, opp, vel in cases:
        d = eng.plan(pose, opp, update_prev=False, opponent_velocities=vel)
        o = MO.plan_motion(cfg, world, pose, opp, vel, want_states=True)
        H.classify_flags(d.flags, o, cfg, counts=counts)
        if d.best_idx != o["best_idx"]:
            counts["argmin_mismatch"] += 1
            gap = abs(float(o["costs"][d.best_idx]) - float(o["costs"][o["best_idx"]]))
            flags_differ = (d.flags[[d.best_idx, o["best_idx"]]] & 0xF) != (o["flags"][[d.best_idx, o["best_idx"]]] & 0xF)
            assert gap < 1e-5 or flags_differ.any(), (d.best_idx, o["best_idx"], gap)
            counts["argmin:cost_gap<1e-5"] += int(gap < 1e-5)
    H.record_parity("moving_opponents_single", counts)
    # batch scenario s == the single query on the same inputs
    K = max(len(c[1]) for c in cases)
    S = len(cases)
    poses = np.array([c[0] for c in cases])
    opp = np.zeros((S, K, 3))
    vel = np.zeros((S, K, 2))
    n_opp = np.zeros(S, np.int32)
    for s, (_, o_, v_) in enumerate(cases):
        opp[s, :len(o_)], vel[s, :len(o_)], n_opp[s] = o_, v_, len(o_)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, opponent_velocities=vel)
    for s in range(S):
        d = eng.plan(poses[s], opp[s, :n_opp[s]], update_prev=False, opponent_velocities=vel[s, :n_opp[s]])
        assert np.array_equal(d.costs, b.costs[s]) and np.array_equal(d.flags, b.flags[s]), s
        assert d.best_idx == b.best_idx[s] and np.array_equal(d.best_traj, b.best_traj[s]), s
        assert d.steer == b.steer_speed[s, 0] and d.speed == b.steer_speed[s, 1], s


# ---- 4. graph replay -----------------------------------------------------------------------------
def test_graph_replay_keeps_static_and_moving_apart(ellipse, corridor):
    eng, _, _ = _pair(ellipse, corridor)
    pose, opp, vel = _crafted(ellipse, 77)
    pose = pose.copy()
    calls = [(None, 1.0), (vel, 1.0), (None, 1.0), (-vel, 1.0), (vel, 1.0), (vel, 4.0), (None, 1.0)]
    slow = pose.copy()
    slow[3] = 0.5
    eng.set_graph(False)
    ref = [eng.plan(slow, opp, update_prev=False, opponent_velocities=v, v_min=vm) for v, vm in calls]
    eng.set_graph(True)
    for _ in range(2):
        for (v, vm), r in zip(calls, ref):
            _assert_same_detail(eng.plan(slow, opp, update_prev=False, opponent_velocities=v, v_min=vm), r)
    assert not np.array_equal(ref[0].flags, ref[1].flags)
    assert not np.array_equal(ref[4].flags, ref[5].flags)   # v_min is part of the answer


def test_bad_motion_arguments(ellipse, corridor):
    import torch
    from f1tenth_planning_b200._lib import F1LError
    eng, _, _ = _pair(ellipse, corridor)
    pose, opp = H.scenario(ellipse, 5, 3)
    for bad in (0.0, -1.0, math.nan, math.inf):
        with pytest.raises(F1LError):
            eng.plan(pose, opp, opponent_velocities=np.zeros((3, 2)), v_min=bad)
    v = np.zeros((3, 2))
    v[1, 0] = math.nan
    with pytest.raises(F1LError):
        eng.plan(pose, opp, opponent_velocities=v)
    with pytest.raises(ValueError):
        eng.plan(pose, opp, opponent_velocities=np.zeros((2, 2)))
    with pytest.raises(ValueError):
        eng.plan(pose, opp, opponent_velocities=np.zeros((3, 2)), rows=(0, 2))
    with pytest.raises(ValueError):
        eng.plan(pose, opp, opponent_velocities=np.zeros((3, 2)), shard=(0, 10))
    poses, opp_b, n_opp = synth.scenario_batch(ellipse, 8, 3, 1)
    vb = np.zeros((8, 3, 2))
    vb[2, 1, 1] = math.inf
    n_opp[2] = 3
    with pytest.raises(F1LError):
        eng.plan_batch(poses, opp_b, n_opp, opponent_velocities=vb)
    with pytest.raises(F1LError):
        eng.plan_batch(poses, opp_b, n_opp, opponent_velocities=np.zeros((8, 3, 2)), v_min=0.0)
    with pytest.raises(ValueError):
        eng.plan_batch(poses, opp_b, n_opp, opponent_velocities=np.zeros((8, 2, 2)))
    dev = torch.device("cuda", eng.device)
    with pytest.raises(ValueError):
        eng.plan_batch_dev(torch.from_numpy(poses).to(dev), torch.from_numpy(opp_b).to(dev),
                           best_idx=torch.empty(8, dtype=torch.int32, device=dev),
                           opponent_velocities=torch.zeros(8, 3, 2, dtype=torch.float32, device=dev))
    # the null velocity pointer with opponents, through the raw ABI
    b = eng._L.f1l_plan_batch_motion
    from f1tenth_planning_b200 import _lib
    call = _lib.batch_call(dict(poses=poses, opp=opp_b, best_idx=np.zeros(8, np.int32)), "host",
                           dict(S=8, K=3, C=eng.n_candidates, M=eng.n_samples), False)
    assert b(eng._h, ctypes.byref(call), None, 1.0) == -1
    f = eng.fleet(poses[:8, :4], group=4)
    with pytest.raises(ValueError):
        f.run(1, predict=True, v_min=0.0)


# ---- 5. fleets ------------------------------------------------------------------------------------
def _fleet_engine(ellipse, corridor):
    eng, _, _ = _pair(ellipse, corridor)
    return eng


def _race_vel(X, status, G, dyn=None):
    """[S,G-1,2] the other cars' velocities in race order, as the step kernel writes them"""
    h = X[:, 2] if dyn is None else X[:, 2] + dyn[:, 2]
    v = np.stack([X[:, 3] * np.cos(h), X[:, 3] * np.sin(h)], axis=1)
    v[(status & 3) != 0] = 0.0
    S = X.shape[0]
    R = v.reshape(S // G, G, 2)
    out = np.zeros((S, G - 1, 2))
    for j in range(G):
        out[j::G] = np.delete(R, j, axis=1)
    return out


@pytest.mark.parametrize("model", ["kinematic", "single_track"])
def test_fleet_predict_teacher_forced(ellipse, corridor, model):
    eng = _fleet_engine(ellipse, corridor)
    S, G = 64, 4
    X0 = _race_poses(ellipse, S, G, 12, 3101, v=5.0)
    veh = Vehicle() if model == "single_track" else None
    f = eng.fleet(X0, group=G, vehicle=veh)
    f.run(25, predict=True)
    n_steps_checked = 0
    for _ in range(3):
        X = f.state.cpu().numpy()
        st = f.status.cpu().numpy()
        P, V = f.prev_theta.cpu().numpy().copy(), f.has_prev.cpu().numpy().copy()
        dyn = f.dyn.cpu().numpy() if veh is not None else None
        tr = _np(f.run(1, trace=True, predict=True))
        b = eng.plan_batch(X, _race_opp(X, G), np.full(S, G - 1, np.int32), want_traj=False, prev_theta=P,
                           has_prev=V, opponent_velocities=_race_vel(X, st, G, dyn))
        assert np.array_equal(tr.state[0], X)
        assert np.array_equal(b.best_idx, tr.best_idx[0])
        assert np.array_equal(b.steer_speed, tr.steer_speed[0])
        n_steps_checked += 1
    # prediction changes the plans of some cars
    fs = eng.fleet(X0, group=G, vehicle=veh)
    fp = eng.fleet(X0, group=G, vehicle=veh)
    a, p = _np(fs.run(20, trace=True)), _np(fp.run(20, trace=True, predict=True))
    assert not np.array_equal(a.best_idx, p.best_idx)


@pytest.mark.parametrize("model", ["kinematic", "single_track"])
def test_fleet_predict_runs_continue(ellipse, corridor, model):
    eng = _fleet_engine(ellipse, corridor)
    S, G = 32, 4
    X0 = _race_poses(ellipse, S, G, 10, 3201, v=6.0)
    veh = Vehicle() if model == "single_track" else None
    one, two = eng.fleet(X0, group=G, vehicle=veh), eng.fleet(X0, group=G, vehicle=veh)
    t1 = _np(one.run(60, trace=True, predict=True))
    t2a = _np(two.run(30, trace=True, predict=True))
    t2b = _np(two.run(30, trace=True, predict=True))
    for k in t1._fields:
        assert np.array_equal(getattr(t1, k), np.concatenate([getattr(t2a, k), getattr(t2b, k)])), k
    for n in ("state", "prev_theta", "has_prev", "status", "progress", "track_i", "track_s"):
        assert np.array_equal(getattr(one, n).cpu().numpy(), getattr(two, n).cpu().numpy()), n
