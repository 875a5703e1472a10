"""Per-scenario previous paths in batch planning (f1l_plan_batch_prev / _dev): scenario s of a
batch gives bit-identically what a single query on the same handle gives after
set_prev_path(prev[s]) (or set_prev_path(None) where has_prev[s] is 0), and update_prev carries
the paths from step to step in place, as plan(update_prev=True) does for one car."""
import ctypes
import os

import numpy as np
import pytest

from f1tenth_planning_b200 import LatticePlanner, synth
from oracle import c_oracle as co
from tests import helpers as H

pytestmark = pytest.mark.gpu

OFF_TRACK = np.array([0.0, 0.0, 0.3, 3.0])   # centre of the oval: no lookahead intersection
NUDGE = np.array([0.05, 0.02, 0.01, 0.0])
CONFIGS = [{}, dict(n_samples=200, n_shift=2, n_cull=3)]
DT, WHEELBASE = 0.01, 0.33


def _pair(ellipse, corridor, **cfg):
    la, wd = synth.goal_grid(4)
    return H.make_pair(ellipse, la, wd, grid=corridor, kappa_max=3.0, **cfg)


def _paths(eng, poses, opp, n_opp):
    """previous paths from a first batch: the theta columns of its best trajectories, with every
    third scenario marked as having none"""
    b0 = eng.plan_batch(poses, opp, n_opp)
    P = np.ascontiguousarray(b0.best_traj[:, :, 2])
    V = np.ones(poses.shape[0], np.uint8)
    V[::3] = 0
    return P, V


def _single(eng, pose, opp, prev):
    eng.set_prev_path(prev)
    return eng.plan(pose, opp, update_prev=False)


def _assert_same(d, b, s):
    assert np.array_equal(d.costs, b.costs[s]), s
    assert np.array_equal(d.flags, b.flags[s]), s
    assert d.best_idx == b.best_idx[s], s
    assert np.float32(d.best_cost) == b.best_cost[s], s
    assert np.array_equal(d.best_traj, b.best_traj[s]), s
    assert d.steer == b.steer_speed[s, 0] and d.speed == b.steer_speed[s, 1], s


@pytest.mark.parametrize("cfg", CONFIGS, ids=["m100", "m200"])
def test_batch_prev_equals_single_query(ellipse, corridor, cfg):
    eng, _, _ = _pair(ellipse, corridor, **cfg)
    S, K = 96, 8
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, K, 1004)
    P, V = _paths(eng, poses, opp, n_opp)
    poses = poses + NUDGE
    # the handle's own previous path must not leak into the batch
    eng.set_prev_path(P[1])
    P0, V0 = P.copy(), V.copy()
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, prev_theta=P, has_prev=V)
    assert np.array_equal(P, P0) and np.array_equal(V, V0)   # read only without update_prev
    ref = eng.plan_batch(poses, opp, n_opp, want_flags=True)
    live = 0
    for s in range(S):
        d = _single(eng, poses[s], opp[s, :n_opp[s]], P[s] if V[s] else None)
        _assert_same(d, b, s)
        if not V[s]:
            assert np.array_equal(b.costs[s], ref.costs[s]) and np.array_equal(b.best_traj[s], ref.best_traj[s])
        elif np.isfinite(ref.costs[s]).any():
            assert not np.array_equal(b.costs[s], ref.costs[s]), s   # the similarity term is live
            live += 1
    assert live > 20


def test_batch_prev_matches_oracle(ellipse, corridor):
    eng, cfg, world = _pair(ellipse, corridor)
    S, K = 96, 8
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, K, 1004)
    P, V = _paths(eng, poses, opp, n_opp)
    poses = poses + NUDGE
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, prev_theta=P, has_prev=V)
    keys = ("costs", "best_idx", "best_cost", "best_traj", "steer_speed")
    o = {k: [] for k in keys}
    for s in range(S):
        world.set_prev(P[s] if V[s] else None)
        r = co.plan(cfg, world, poses[s], opp[s, :n_opp[s]])
        for k in keys:
            o[k].append(r[k] if k != "steer_speed" else [r["steer"], r["speed"]])
    world.set_prev(None)
    o = {k: np.array(v) for k, v in o.items()}
    fin = np.isfinite(o["costs"]) & np.isfinite(b.costs)
    assert fin.sum() > 200
    assert H.close(b.costs[fin], o["costs"][fin]).all()
    fin_mismatch = (np.isfinite(o["costs"]) != np.isfinite(b.costs)).mean()
    assert fin_mismatch < 0.01
    agree = b.best_idx == o["best_idx"]
    for s in np.nonzero(~agree)[0]:
        gap = abs(float(o["costs"][s, b.best_idx[s]]) - float(o["best_cost"][s]))
        assert gap < 1e-5, (s, gap)
    ok = agree & np.isfinite(o["best_cost"])
    assert ok.sum() > 50
    assert H.close(b.best_traj[ok], o["best_traj"][ok], scale=H.traj_scale(o["best_traj"][ok])).all()
    assert H.close(b.steer_speed[ok], o["steer_speed"][ok], 1e-4, 1e-4).all()
    H.record_parity("batch_prev_96_scenarios", {
        "scenarios": S, "with_prev": int(V.sum()), "finite_both": int(fin.sum()),
        "finiteness_mismatch_frac": float(fin_mismatch), "argmin_mismatch": int((~agree).sum()),
        "cost_rel_err_max": float((np.abs(b.costs[fin] - o["costs"][fin])
                                   / (H.ABS / H.REL + np.abs(o["costs"][fin]))).max())})


def test_update_prev_in_place(ellipse, corridor):
    eng, _, _ = _pair(ellipse, corridor)
    S, K, off = 96, 8, 5
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, K, 1004)
    P, V = _paths(eng, poses, opp, n_opp)
    poses = poses + NUDGE
    poses[off] = OFF_TRACK
    Pb, Vb = P.copy(), V.astype(bool)
    # the handle's single-query previous path before and after the batch
    eng.set_prev_path(P[2])
    probe = poses[7]
    before = eng.plan(probe, update_prev=False)
    b = eng.plan_batch(poses, opp, n_opp, prev_theta=P, has_prev=Vb, update_prev=True)
    after = eng.plan(probe, update_prev=False)
    assert np.array_equal(before.costs, after.costs) and before.best_idx == after.best_idx
    assert np.array_equal(P, b.best_traj[:, :, 2]) and Vb.all()
    assert not np.isfinite(b.best_cost[off]) and b.best_idx[off] == 0
    # the off-track, all-infeasible scenario stores what plan(update_prev=True) stores
    eng.set_prev_path(Pb[off] if V[off] else None)
    d = eng.plan(OFF_TRACK, update_prev=True)
    assert d.no_feasible and np.array_equal(P[off], d.best_traj[:, 2])
    # ... and the next step from there agrees both ways
    nxt = poses.copy()
    nxt[off] = poses[off + 1]
    b2 = eng.plan_batch(nxt, opp, n_opp, want_flags=True, prev_theta=P, has_prev=Vb)
    d2 = eng.plan(nxt[off], opp[off, :n_opp[off]], update_prev=False)
    assert np.isfinite(d2.best_cost)
    _assert_same(d2, b2, off)


@pytest.mark.parametrize("S", [4096, 20000], ids=["equal_chunks", "tapered_tail"])
def test_host_pipeline_matches_device_api(ellipse, corridor, S):
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 8, 1006)
    P, V = _paths(eng, poses, opp, n_opp)
    poses = poses + NUDGE
    dev = torch.device("cuda", eng.device)
    tP, tV = torch.from_numpy(P).to(dev), torch.from_numpy(V).to(dev)
    C, M = eng.n_candidates, eng.n_samples
    out = dict(best_idx=torch.empty(S, dtype=torch.int32, device=dev),
               best_cost=torch.empty(S, dtype=torch.float32, device=dev),
               best_traj=torch.empty(S, M, 4, dtype=torch.float32, device=dev),
               costs=torch.empty(S, C, dtype=torch.float32, device=dev),
               flags=torch.empty(S, C, dtype=torch.uint8, device=dev),
               steer_speed=torch.empty(S, 2, dtype=torch.float64, device=dev))
    eng.plan_batch_dev(torch.from_numpy(poses).to(dev), torch.from_numpy(opp).to(dev),
                       torch.from_numpy(n_opp).to(dev), prev_theta=tP, has_prev=tV, update_prev=True,
                       **out)
    torch.cuda.synchronize(dev)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, prev_theta=P, has_prev=V, update_prev=True)
    for k, v in out.items():
        assert np.array_equal(v.cpu().numpy(), getattr(b, k)), k
    assert np.array_equal(tP.cpu().numpy(), P) and np.array_equal(tV.cpu().numpy(), V)
    assert V.all() and np.array_equal(P, b.best_traj[:, :, 2])


def _spielberg(golden_spielberg):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "maps.npz"))
    w = int(g["spielberg_shape"][1])
    occ = np.unpackbits(g["spielberg_bits"], axis=1)[:, :w]
    return golden_spielberg["waypoints"], (occ, tuple(g["spielberg_origin"]), float(g["spielberg_res"]))


def test_closed_loop_batch_rollout(golden_spielberg):
    """32 cars on the Spielberg raceline, 200 steps of the kinematic bicycle of
    test_gpu_closed_loop, driven by one batch call per step that carries every car's previous
    path; a single-query handle plans each car in lockstep with its own carried path."""
    wp, grid = _spielberg(golden_spielberg)
    pl = LatticePlanner(wheelbase=WHEELBASE, waypoints=wp)
    pl.set_map(*grid)
    pl.set_goal_grid(np.linspace(0.8, 3.0, 8), np.linspace(-0.6, 0.6, 9))
    eng = pl.engine
    S, N_STEPS, v_cap, dev_max = 32, 200, 5.0, 0.8
    start = np.linspace(0, wp.shape[0], S, endpoint=False).astype(int)
    X = np.stack([wp[start, 0], wp[start, 1], wp[start, 3], np.full(S, 5.0)], axis=1)
    P = np.zeros((S, eng.n_samples), np.float32)
    V = np.zeros(S, np.uint8)
    own = [None] * S
    path = [[] for _ in range(S)]
    reset = {100: (3, 17)}
    for k in range(N_STEPS):
        for c in reset.get(k, ()):   # a fresh car elsewhere on the raceline, no previous path
            i = (start[c] + wp.shape[0] // (2 * S)) % wp.shape[0]
            X[c] = [wp[i, 0], wp[i, 1], wp[i, 3], 5.0]
            V[c] = 0
            own[c] = None
            path[c] = []
        b = pl.plan_batch(X, prev_theta=P, has_prev=V, update_prev=True)
        assert V.all() and np.isfinite(b.best_cost).all(), k
        for c in range(S):
            eng.set_prev_path(own[c])
            d = eng.plan(X[c], update_prev=True)
            own[c] = d.best_traj[:, 2].copy()
            assert d.best_idx == b.best_idx[c] and np.float32(d.best_cost) == b.best_cost[c], (k, c)
            assert np.array_equal(P[c], own[c]), (k, c)
        steer = np.clip(b.steer_speed[:, 0], -0.4189, 0.4189)
        X[:, 3] += np.clip(np.minimum(b.steer_speed[:, 1], v_cap) - X[:, 3], -9.51 * DT, 9.51 * DT)
        X[:, 0] += X[:, 3] * np.cos(X[:, 2]) * DT
        X[:, 1] += X[:, 3] * np.sin(X[:, 2]) * DT
        X[:, 2] += X[:, 3] / WHEELBASE * np.tan(steer) * DT
        for c in range(S):
            path[c].append(X[c, :2].copy())
    worst = 0.0
    for c in range(S):
        p = np.array(path[c])
        assert np.hypot(*(p[-1] - p[0])) > 3.0, c
        worst = max(worst, max(co.nearest_point(q, wp[:, :2])[1] for q in p[::20]))
    assert worst < dev_max, worst


def test_device_resident_loop(ellipse, corridor):
    """plan_batch_dev with the paths as CUDA tensors, the bicycle stepped in torch on the same
    stream; every step checked against plan_batch on the state downloaded before it."""
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    S, K = 256, 8
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, K, 1007)
    P, V = _paths(eng, poses, opp, n_opp)
    dev = torch.device("cuda", eng.device)
    stream = torch.cuda.Stream(dev)
    M, C = eng.n_samples, eng.n_candidates
    with torch.cuda.stream(stream):
        tX, to, tn = (torch.from_numpy(a).to(dev) for a in (poses, opp, n_opp))
        tP, tV = torch.from_numpy(P).to(dev), torch.from_numpy(V).to(dev)
        idx = torch.empty(S, dtype=torch.int32, device=dev)
        cost = torch.empty(S, dtype=torch.float32, device=dev)
        costs = torch.empty(S, C, dtype=torch.float32, device=dev)
        ss = torch.empty(S, 2, dtype=torch.float64, device=dev)
        for k in range(20):
            X0, P0, V0 = tX.cpu().numpy(), tP.cpu().numpy(), tV.cpu().numpy()
            eng.plan_batch_dev(tX, to, tn, best_idx=idx, best_cost=cost, costs=costs, steer_speed=ss,
                               stream=stream.cuda_stream, prev_theta=tP, has_prev=tV, update_prev=True)
            steer = ss[:, 0].clamp(-0.4189, 0.4189)
            v = tX[:, 3] + (torch.minimum(ss[:, 1], torch.full_like(ss[:, 1], 5.0)) - tX[:, 3]).clamp(
                -9.51 * DT, 9.51 * DT)
            tX = torch.stack([tX[:, 0] + v * torch.cos(tX[:, 2]) * DT, tX[:, 1] + v * torch.sin(tX[:, 2]) * DT,
                              tX[:, 2] + v / WHEELBASE * torch.tan(steer) * DT, v], dim=1)
            b = eng.plan_batch(X0, opp, n_opp, prev_theta=P0, has_prev=V0, update_prev=True)
            assert np.array_equal(idx.cpu().numpy(), b.best_idx), k
            assert np.array_equal(costs.cpu().numpy(), b.costs), k
            assert np.array_equal(ss.cpu().numpy(), b.steer_speed), k
            assert np.array_equal(tP.cpu().numpy(), P0) and np.array_equal(tV.cpu().numpy(), V0), k
    assert V0.all()


def test_bad_prev_arguments_are_rejected(ellipse, corridor):
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    S, M = 8, eng.n_samples
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 2, 1008)
    good = np.zeros((S, M), np.float32)
    V = np.ones(S, np.uint8)
    for bad in (np.zeros((S, M + 1), np.float32), np.zeros((S, M), np.float64),
                np.zeros((S, 2 * M), np.float32)[:, ::2], np.asfortranarray(good),
                np.zeros(S * M, np.float32), list(good)):
        with pytest.raises(ValueError):
            eng.plan_batch(poses, opp, n_opp, prev_theta=bad, has_prev=V)
    for bad in (np.ones(S, np.int32), np.ones(S + 1, np.uint8), np.ones(2 * S, np.uint8)[::2]):
        with pytest.raises(ValueError):
            eng.plan_batch(poses, opp, n_opp, prev_theta=good, has_prev=bad)
    ro = good.copy()
    ro.flags.writeable = False
    with pytest.raises(ValueError):
        eng.plan_batch(poses, opp, n_opp, prev_theta=ro, update_prev=True)
    with pytest.raises(ValueError):
        eng.plan_batch(poses, opp, n_opp, has_prev=V)
    with pytest.raises(ValueError):
        eng.plan_batch(poses, opp, n_opp, update_prev=True)
    eng.plan_batch(poses, opp, n_opp, prev_theta=ro)   # read-only input is fine without update_prev

    dev = torch.device("cuda", eng.device)
    tX, to, tn = (torch.from_numpy(a).to(dev) for a in (poses, opp, n_opp))
    tgood, tV = torch.zeros(S, M, device=dev), torch.ones(S, dtype=torch.uint8, device=dev)
    for bad in (torch.zeros(S, M + 1, device=dev), torch.zeros(S, M, dtype=torch.float64, device=dev),
                torch.zeros(M, S, device=dev).t(), torch.zeros(S, M), good):
        with pytest.raises(ValueError):
            eng.plan_batch_dev(tX, to, tn, prev_theta=bad, has_prev=tV)
    with pytest.raises(ValueError):
        eng.plan_batch_dev(tX, to, tn, prev_theta=tgood, has_prev=torch.ones(S, dtype=torch.int32, device=dev))
    with pytest.raises(ValueError):
        eng.plan_batch_dev(tX, to, tn, has_prev=tV)
    with pytest.raises(ValueError):
        eng.plan_batch_dev(tX, to, tn, update_prev=True)

    # the raw ABI: has_prev or update_prev without prev_theta
    L, vp = eng._L, ctypes.c_void_p
    out = np.zeros(S, np.int32)
    p, v = vp(poses.ctypes.data), vp(V.ctypes.data)
    assert L.f1l_plan_batch_prev(eng._h, p, None, None, S, 0, None, v, 0, vp(out.ctypes.data),
                                 None, None, None, None, None) == -1
    assert L.f1l_plan_batch_prev(eng._h, p, None, None, S, 0, None, None, 1, vp(out.ctypes.data),
                                 None, None, None, None, None) == -1
    assert L.f1l_plan_batch_prev_dev(eng._h, vp(tX.data_ptr()), None, None, S, 0, None, vp(tV.data_ptr()),
                                     0, None, None, None, None, None, None, None) == -1
    assert L.f1l_plan_batch_prev_dev(eng._h, vp(tX.data_ptr()), None, None, S, 0, None, None, 1,
                                     None, None, None, None, None, None, None) == -1
