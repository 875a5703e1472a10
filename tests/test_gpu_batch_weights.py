"""Cost weights per scenario and per-term costs in batch planning (f1l_plan_batch_call / _dev) and in
closed-loop rollouts (f1l_rollout_weights_dev): scenario s with weights w[s] gives bit-identically
what a single query on the same handle gives after configure(weights=w[s]), and with the config's
weights (or none) what the batch gave before."""
import ctypes

import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from oracle import c_oracle as co
from tests import helpers as H
from tests.test_gpu_batch_prev import CONFIGS, NUDGE, _assert_same, _pair, _paths
from tests.test_gpu_rollout import _ellipse_engine, _np, _race_opp, _race_poses, _spielberg_engine

pytestmark = pytest.mark.gpu

FIELDS = ("best_idx", "best_cost", "best_traj", "costs", "flags", "steer_speed")


def _weight_rows(default, S, seed):
    """the defaults, the one-hot rows (deviation-only, similarity-only, ...), a zero in each term in
    turn, rows that do not sum to 1, then random rows up to S"""
    d = np.asarray(default, np.float64)
    rows = [d]
    rows += list(np.eye(5))
    for k in range(5):
        r = d.copy()
        r[k] = 0.0
        rows.append(r)
    rows += [3.0 * d, 0.1 * d, np.array([2.0, 0.5, 4.0, 0.0, 7.0]), np.array([0.0, 0.0, 0.0, 5.0, 5.0])]
    rng = np.random.default_rng(seed)
    rows += list(rng.uniform(0.0, 2.0, (S - len(rows), 5)))
    return np.array(rows).astype(np.float32)


def _scenarios(eng, ellipse, S, seed):
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 8, seed)
    P, V = _paths(eng, poses, opp, n_opp)
    return poses + NUDGE, opp, n_opp, P, V


@pytest.mark.parametrize("cfg", CONFIGS, ids=["m100", "m200"])
@pytest.mark.parametrize("with_prev", [False, True], ids=["no_prev", "prev"])
def test_weights_equal_single_queries(ellipse, corridor, cfg, with_prev):
    eng, _, _ = _pair(ellipse, corridor, **cfg)
    S = 96
    poses, opp, n_opp, P, V = _scenarios(eng, ellipse, S, 1104)
    prev = dict(prev_theta=P, has_prev=V) if with_prev else {}
    default = list(eng.config.weights)
    W = _weight_rows(default, S, 7)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, weights=W, want_terms=True, **prev)
    ref = eng.plan_batch(poses, opp, n_opp, want_flags=True, **prev)
    new_idx = new_costs = 0
    for s in range(S):
        eng.configure(weights=W[s].astype(np.float64))
        eng.set_prev_path(P[s] if with_prev and V[s] else None)
        d = eng.plan(poses[s], opp[s, :n_opp[s]], update_prev=False)
        _assert_same(d, b, s)
        assert np.array_equal(d.terms, b.terms[s]), s
        new_idx += int(b.best_idx[s] != ref.best_idx[s])
        new_costs += int(not np.array_equal(b.costs[s], ref.costs[s]))
    eng.configure(weights=default)
    # the weights are live: most scenarios' costs and some of their argmins change
    assert new_costs >= S // 2 and new_idx >= 5, (new_costs, new_idx)


def test_config_weights_broadcast_change_nothing(ellipse, corridor):
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    S = 256
    poses, opp, n_opp, P, V = _scenarios(eng, ellipse, S, 1105)
    W = np.tile(np.array(list(eng.config.weights), np.float32), (S, 1))
    a = eng.plan_batch(poses, opp, n_opp, want_flags=True)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, weights=W)
    for k in FIELDS:
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    dev = torch.device("cuda", eng.device)
    C, M = eng.n_candidates, eng.n_samples
    tX, to, tn = (torch.from_numpy(x).to(dev) for x in (poses, opp, n_opp))
    outs = []
    for w in (None, torch.from_numpy(W).to(dev)):
        o = dict(best_idx=torch.empty(S, dtype=torch.int32, device=dev),
                 best_cost=torch.empty(S, dtype=torch.float32, device=dev),
                 best_traj=torch.empty(S, M, 4, dtype=torch.float32, device=dev),
                 costs=torch.empty(S, C, dtype=torch.float32, device=dev),
                 flags=torch.empty(S, C, dtype=torch.uint8, device=dev),
                 steer_speed=torch.empty(S, 2, dtype=torch.float64, device=dev))
        eng.plan_batch_dev(tX, to, tn, weights=w, **o)
        torch.cuda.synchronize(dev)
        outs.append({k: v.cpu().numpy() for k, v in o.items()})
    for k in FIELDS:
        assert np.array_equal(outs[0][k], outs[1][k]), k
        assert np.array_equal(outs[0][k], getattr(a, k)), k


@pytest.mark.parametrize("prune", [0, 1])
def test_terms_equal_plan_detailed_and_weighted_sum(ellipse, corridor, prune):
    eng, _, _ = _pair(ellipse, corridor, prune_window=prune)
    S = 96
    poses, opp, n_opp, P, V = _scenarios(eng, ellipse, S, 1106)
    W = _weight_rows(list(eng.config.weights), S, 8)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, weights=W, want_terms=True,
                       prev_theta=P, has_prev=V)
    default = list(eng.config.weights)
    n_fin = 0
    for s in range(S):
        eng.configure(weights=W[s].astype(np.float64))
        eng.set_prev_path(P[s] if V[s] else None)
        d = eng.plan(poses[s], opp[s, :n_opp[s]], update_prev=False)
        assert np.array_equal(d.terms, b.terms[s]), s
        fin = np.isfinite(b.costs[s])
        n_fin += int(fin.sum())
        t = b.terms[s][fin].astype(np.float64)
        want = t @ W[s].astype(np.float64)
        assert np.allclose(b.costs[s][fin], want, rtol=1e-6, atol=1e-6), s
    eng.configure(weights=default)
    assert n_fin > 400


def test_host_pipeline_matches_device_call(ellipse, corridor):
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    S = 20000
    poses, opp, n_opp, P, V = _scenarios(eng, ellipse, S, 1107)
    W = np.random.default_rng(9).uniform(0.0, 2.0, (S, 5)).astype(np.float32)
    dev = torch.device("cuda", eng.device)
    C, M = eng.n_candidates, eng.n_samples
    tP, tV = torch.from_numpy(P).to(dev), torch.from_numpy(V).to(dev)
    out = dict(best_idx=torch.empty(S, dtype=torch.int32, device=dev),
               best_cost=torch.empty(S, dtype=torch.float32, device=dev),
               best_traj=torch.empty(S, M, 4, dtype=torch.float32, device=dev),
               costs=torch.empty(S, C, dtype=torch.float32, device=dev),
               flags=torch.empty(S, C, dtype=torch.uint8, device=dev),
               steer_speed=torch.empty(S, 2, dtype=torch.float64, device=dev),
               terms=torch.empty(S, C, 5, dtype=torch.float32, device=dev))
    eng.plan_batch_dev(torch.from_numpy(poses).to(dev), torch.from_numpy(opp).to(dev),
                       torch.from_numpy(n_opp).to(dev), prev_theta=tP, has_prev=tV, update_prev=True,
                       weights=torch.from_numpy(W).to(dev), **out)
    torch.cuda.synchronize(dev)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, prev_theta=P, has_prev=V, update_prev=True,
                       weights=W, want_terms=True)
    for k, v in out.items():
        assert np.array_equal(v.cpu().numpy(), getattr(b, k)), k
    assert np.array_equal(tP.cpu().numpy(), P) and np.array_equal(tV.cpu().numpy(), V)
    assert V.all() and np.array_equal(P, b.best_traj[:, :, 2])


def test_weights_match_oracle(ellipse, corridor):
    eng, _, world = _pair(ellipse, corridor)
    S = 48
    poses, opp, n_opp, P, V = _scenarios(eng, ellipse, S, 1108)
    W = _weight_rows(list(eng.config.weights), S, 10)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True, prev_theta=P, has_prev=V, weights=W)
    default = list(eng.config.weights)
    keys = ("costs", "best_idx", "best_cost")
    o = {k: [] for k in keys}
    for s in range(S):
        eng.configure(weights=W[s].astype(np.float64))
        cfg = H.oracle_config_from_engine(eng)
        world.set_prev(P[s] if V[s] else None)
        r = co.plan(cfg, world, poses[s], opp[s, :n_opp[s]])
        for k in keys:
            o[k].append(r[k])
    world.set_prev(None)
    eng.configure(weights=default)
    o = {k: np.array(v) for k, v in o.items()}
    fin = np.isfinite(o["costs"]) & np.isfinite(b.costs)
    assert fin.sum() > 100
    assert H.close(b.costs[fin], o["costs"][fin]).all()
    fin_mismatch = (np.isfinite(o["costs"]) != np.isfinite(b.costs)).mean()
    assert fin_mismatch < 0.01
    agree = b.best_idx == o["best_idx"]
    for s in np.nonzero(~agree)[0]:
        gap = abs(float(o["costs"][s, b.best_idx[s]]) - float(o["best_cost"][s]))
        assert gap < 1e-5 * max(1.0, abs(float(o["best_cost"][s]))), (s, gap)
    H.record_parity("batch_weights_48_scenarios", {
        "scenarios": S, "finite_both": int(fin.sum()), "finiteness_mismatch_frac": float(fin_mismatch),
        "argmin_mismatch": int((~agree).sum()),
        "cost_rel_err_max": float((np.abs(b.costs[fin] - o["costs"][fin])
                                   / (H.ABS / H.REL + np.abs(o["costs"][fin]))).max())})


def _fleet_state(f):
    return {n: getattr(f, n).cpu().numpy() for n in
            ("state", "prev_theta", "has_prev", "status", "progress", "track_i", "track_s")}


def test_rollout_weights_null_and_config_equal_plain_rollout(ellipse, corridor):
    import torch
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 5, 2101)
    Wc = np.tile(np.array(list(eng.config.weights), np.float32), (S, 1))
    plain = eng.fleet(X0, group=G)
    tr0 = _np(plain.run(40, substeps=2, trace=True))
    for w in (None, Wc):
        f = eng.fleet(X0, group=G, weights=w)
        tr = _np(f.run(40, substeps=2, trace=True))
        for k in tr._fields:
            assert np.array_equal(getattr(tr, k), getattr(tr0, k)), k
        for k, v in _fleet_state(f).items():
            assert np.array_equal(v, _fleet_state(plain)[k]), k
    assert isinstance(eng.fleet(X0, group=G, weights=Wc).weights, torch.Tensor)


def test_rollout_weights_teacher_forced_spielberg(golden_spielberg):
    eng, wp, grid = _spielberg_engine(golden_spielberg)
    S, G = 32, 4
    X0 = _race_poses(wp, S, G, 6, 2111)
    W = _weight_rows(list(eng.config.weights), S, 12)
    fleet = eng.fleet(X0, group=G, weights=W)
    tr = _np(fleet.run(40, substeps=5, v_max=5.0, trace=True))
    P = np.zeros((S, eng.n_samples), np.float32)
    V = np.zeros(S, np.uint8)
    for k in range(tr.best_idx.shape[0]):
        X = tr.state[k]
        b = eng.plan_batch(X, _race_opp(X, G), np.full(S, G - 1, np.int32), want_traj=False,
                           want_costs=False, prev_theta=P, has_prev=V, update_prev=True, weights=W)
        assert np.array_equal(b.best_idx, tr.best_idx[k]), k
        assert np.array_equal(b.steer_speed, tr.steer_speed[k]), k


def test_rollout_weights_diverge_and_continue(ellipse, corridor):
    eng, wp, grid = _ellipse_engine(ellipse, corridor)
    S, G = 32, 4
    X1 = _race_poses(wp, S // 2, G, 5, 2121)
    X0 = np.concatenate([X1, X1])   # races r and r + 4 start from identical poses
    d = np.array(list(eng.config.weights), np.float32)
    W = np.concatenate([np.tile(d, (S // 2, 1)), np.tile(np.array([0.0, 0.0, 0.0, 0.0, 1.0], np.float32),
                                                          (S // 2, 1))])
    a, b = eng.fleet(X0, group=G, weights=W), eng.fleet(X0, group=G, weights=W)
    tr = _np(a.run(30, substeps=2, trace=True))
    a.run(30, substeps=2)
    b.run(60, substeps=2)
    for k, v in _fleet_state(a).items():
        assert np.array_equal(v, _fleet_state(b)[k]), k
    diff = (tr.best_idx[:, :S // 2] != tr.best_idx[:, S // 2:]).any(axis=0)
    assert diff.sum() >= S // 4, diff
    st = a.state.cpu().numpy()
    assert not np.array_equal(st[:S // 2], st[S // 2:])


def test_bad_weights_and_terms_are_rejected(ellipse, corridor):
    import torch
    eng, _, _ = _pair(ellipse, corridor)
    S, C = 8, eng.n_candidates
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 2, 1109)
    for bad in (np.ones((S, 4), np.float32), np.ones((S + 1, 5), np.float32), np.ones(S * 5, np.float32),
                np.ones((S, 5), np.int32), [[1, 1, 1, 1, 1]] * S):
        with pytest.raises(ValueError):
            eng.plan_batch(poses, opp, n_opp, weights=bad)
    eng.plan_batch(poses, opp, n_opp, weights=np.ones((5, S), np.float64).T)   # converted
    for bad in (np.zeros((S, C, 4), np.float32), np.zeros((S, C, 5), np.float64),
                np.asfortranarray(np.zeros((S, C, 5), np.float32))):
        with pytest.raises(ValueError):
            eng.plan_batch(poses, opp, n_opp, want_terms=True, out={"terms": bad})
    dev = torch.device("cuda", eng.device)
    tX, to, tn = (torch.from_numpy(a).to(dev) for a in (poses, opp, n_opp))
    good_w = torch.ones(S, 5, device=dev)
    for bad in (torch.ones(S, 4, device=dev), torch.ones(S, 5, dtype=torch.float64, device=dev),
                torch.ones(5, S, device=dev).t(), torch.ones(S, 5), np.ones((S, 5), np.float32)):
        with pytest.raises(ValueError):
            eng.plan_batch_dev(tX, to, tn, weights=bad)
    for bad in (torch.zeros(S, C, 4, device=dev), torch.zeros(S, C, 5, dtype=torch.float64, device=dev),
                torch.zeros(S, 5, C, device=dev).transpose(1, 2), torch.zeros(S, C, 5)):
        with pytest.raises(ValueError):
            eng.plan_batch_dev(tX, to, tn, weights=good_w, terms=bad)
    with pytest.raises(ValueError):
        eng.fleet(poses, group=1, weights=np.ones((S, 4)))
    f = eng.fleet(poses, group=1, weights=np.ones((S, 5)))
    f.weights = torch.ones(S, 5, dtype=torch.float64, device=dev)
    with pytest.raises(ValueError):
        f.run(1)

    # the raw ABI
    from f1tenth_planning_b200 import _lib
    L = eng._L
    V = np.ones(S, np.uint8)
    out = np.zeros(S, np.int32)
    p = tX.data_ptr()
    assert L.f1l_plan_batch_call_dev(eng._h, None, None) == -1
    assert L.f1l_plan_batch_call(eng._h, None) == -1
    b = _lib.BatchCall(poses=poses.ctypes.data, n_scenarios=S, has_prev=V.ctypes.data,
                       best_idx=out.ctypes.data)
    assert L.f1l_plan_batch_call(eng._h, ctypes.byref(b)) == -1
    tV = torch.ones(S, dtype=torch.uint8, device=dev)
    b = _lib.BatchCall(poses=p, n_scenarios=S, has_prev=tV.data_ptr())
    assert L.f1l_plan_batch_call_dev(eng._h, ctypes.byref(b), None) == -1
    for kw in (dict(n_scenarios=0), dict(n_scenarios=S, max_opp=17, opp=to.data_ptr()),
               dict(n_scenarios=S, max_opp=-1), dict(n_scenarios=S, update_prev=1)):
        b = _lib.BatchCall(poses=p, **kw)
        assert L.f1l_plan_batch_call_dev(eng._h, ctypes.byref(b), None) == -1, kw
    torch.cuda.synchronize(dev)
