"""BASELINE.json's full sizes through size-independent properties plus oracle samples:
config 4 (10^5 scenarios x 28 candidates) and config 5 (65 536 candidates x 200 samples)."""
import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from oracle import c_oracle as co
from tests import helpers as H

pytestmark = pytest.mark.gpu


def test_config4_hundred_thousand_scenarios(ellipse, corridor):
    la, wd = synth.goal_grid(4)
    eng, cfg, world = H.make_pair(ellipse, la, wd, grid=corridor, kappa_max=0.0, use_device_lut=False)
    S, K = 100000, 8
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, K, 1004)
    b = eng.plan_batch(poses, opp, n_opp, want_flags=True)
    # argmin semantics at full size: first minimum of the cost vector, +inf rows -> index 0
    am = np.argmin(b.costs, axis=1)
    assert np.array_equal(b.best_idx, am.astype(np.int32))
    assert np.array_equal(b.best_cost, b.costs[np.arange(S), am])
    valid = (b.flags & 1) != 0
    hit = (b.flags & 6) != 0
    assert np.array_equal(np.isfinite(b.costs), valid & ~hit)     # cost finite <=> valid and free
    assert 0.85 < valid.mean() <= 1.0 and 0.02 < hit[valid].mean() < 0.5
    feasible = np.isfinite(b.best_cost)
    assert np.isfinite(b.best_traj[feasible]).all()
    # trajectories start at the vehicle origin and end at the selected goal
    assert np.abs(b.best_traj[feasible][:, 0, :3]).max() == 0.0
    # scenario sharding: any block evaluated alone gives the same answers (weak-scaling shards)
    for lo, hi in ((0, 12500), (50000, 62500), (87500, 100000)):
        part = eng.plan_batch(poses[lo:hi], opp[lo:hi], n_opp[lo:hi], want_flags=True)
        assert np.array_equal(part.best_idx, b.best_idx[lo:hi])
        assert np.array_equal(part.costs, b.costs[lo:hi])
        assert np.array_equal(part.best_traj, b.best_traj[lo:hi])
    # idempotence
    b2 = eng.plan_batch(poses, opp, n_opp, want_flags=True)
    assert np.array_equal(b2.costs, b.costs) and np.array_equal(b2.best_traj, b.best_traj)
    # oracle (seeded from its OWN float64 LUT, not the device's) on 4096 scenarios: every flag,
    # finiteness and argmin mismatch must fall into a margin class (helpers.compare_batch); the
    # observed counts go to the parity log
    sub = np.sort(np.random.default_rng(0).choice(S, 4096, replace=False))
    counts = H.compare_batch(b, sub, poses, opp, n_opp, cfg, world)
    assert counts["flag_mismatch_candidates"] <= 0.002 * counts["candidates"], counts
    assert counts["argmin_mismatch"] <= 0.01 * counts["scenarios"], counts
    H.record_parity("c4_full_size_oracle_own_lut", counts)


def test_config4_collision_flags_bit_exact_mirror(ellipse, corridor):
    """Teacher-forced at C4 scale: on the device's own float32 states the float32 mirror of the
    collision predicate reproduces the opponent / map flags of 1024 scenarios x 28 candidates
    with ZERO mismatches (the float64 comparison above can only classify boundary cases)."""
    la, wd = synth.goal_grid(4)
    eng, cfg, world = H.make_pair(ellipse, la, wd, grid=corridor, kappa_max=0.0)
    poses, opp, n_opp = synth.scenario_batch(ellipse, 100000, 8, 1004)
    hl, hw = np.float32(0.5 * cfg.car_length), np.float32(0.5 * cfg.car_width)
    rc2 = np.float32(4.0 * ((0.5 * cfg.car_length) ** 2 + (0.5 * cfg.car_width) ** 2))
    n_valid = n_hit = mism = 0
    for s in np.random.default_rng(1).choice(100000, 1024, replace=False):
        d = eng.plan(poses[s], opp[s, :n_opp[s]], update_prev=False, want_states=True, want_headings=True)
        f, i = eng.debug_query_ctx()
        mirror = co.collide_f32(d.states, d.headings, f[8:].reshape(16, 4), int(i[5]), f[2:8],
                                i[0:2], corridor[0], hl, hw, rc2)
        valid = (d.flags & 1) != 0
        mism += int((mirror[valid] != (d.flags[valid] & 6)).sum())
        n_valid += int(valid.sum())
        n_hit += int((mirror[valid] != 0).sum())
    H.record_parity("c4_collision_mirror_f32", {"scenarios": 1024, "valid_candidates": n_valid,
                                                "colliding": n_hit, "flag_mismatches": mism})
    assert mism == 0 and n_valid > 20000 and n_hit > 500


def test_config5_dense_sweep(ellipse, corridor):
    la, wd = synth.goal_grid(5)
    eng, cfg, world = H.make_pair(ellipse, la, wd, grid=corridor, n_samples=200, use_device_lut=False)
    pose, opp = H.scenario(ellipse, 1005, 8)
    d = eng.plan(pose, opp, update_prev=False)
    # 32-candidate chunks, 2048 CTAs against 444 resident: the persistent grid on the wide build
    shape = eng.last_eval_shape()
    assert shape["nw"] == 8 and shape["minb"] == 2, shape
    C = 65536
    assert d.costs.shape == (C,)
    assert d.best_idx == int(np.argmin(d.costs)) and d.best_cost == d.costs[d.best_idx]
    valid = (d.flags & 1) != 0
    assert np.array_equal(np.isfinite(d.costs), valid & ((d.flags & 6) == 0))
    assert valid.sum() > 20000
    # neighbouring goals give neighbouring costs (the cost field is smooth where it is finite)
    grid = d.costs.reshape(256, 256)
    both = np.isfinite(grid[:, 1:]) & np.isfinite(grid[:, :-1])
    assert np.median(np.abs(np.diff(grid, axis=1))[both]) < 5e-3
    # candidate shards reassemble to the full sweep
    best = (np.inf, C)
    for g in range(8):
        lo, hi = g * C // 8, (g + 1) * C // 8
        part = eng.plan(pose, opp, update_prev=False, shard=(lo, hi))
        assert np.array_equal(part.costs[lo:hi], d.costs[lo:hi])
        best = min(best, (float(part.best_cost), int(part.best_idx)))
    assert best[1] == d.best_idx
    # oracle (own float64 LUT) on 8192 candidates of the sweep, 16 slices of 512 spread over the
    # lookahead rows: every mismatch classified, counts to the parity log
    counts = {"candidates": 0}
    err_max = 0.0
    for lo in range(1024, C, C // 16):
        hi = lo + 512
        o = co.plan(cfg, world, pose, opp, c_begin=lo, c_end=hi, want_states=True)
        osl = {k: (v[lo:hi] if isinstance(v, np.ndarray) and v.shape[:1] == (C,) else v) for k, v in o.items()}
        H.classify_flags(d.flags[lo:hi], osl, cfg, counts=counts)
        same = (d.flags[lo:hi] & 0xF) == (osl["flags"] & 0xF)
        fin = np.isfinite(osl["costs"]) & np.isfinite(d.costs[lo:hi])
        assert (np.isfinite(osl["costs"]) == np.isfinite(d.costs[lo:hi]))[same].all()
        assert H.close(d.costs[lo:hi][fin], osl["costs"][fin]).all()
        if fin.any():
            err_max = max(err_max, float((np.abs(d.costs[lo:hi][fin] - osl["costs"][fin]) /
                                          (H.ABS / H.REL + np.abs(osl["costs"][fin]))).max()))
        counts["candidates"] += hi - lo
        counts["flag_mismatch_candidates"] = counts.get("flag_mismatch_candidates", 0) + int((~same).sum())
    counts["cost_rel_err_max"] = err_max
    assert counts["candidates"] >= 8192
    assert counts["flag_mismatch_candidates"] <= 0.004 * counts["candidates"], counts
    H.record_parity("c5_dense_sweep_oracle_own_lut", counts)


def test_config2_full_size_properties(ellipse):
    """10^5 poses on the 2k-waypoint track: permutation invariance and block consistency"""
    from f1tenth_planning_b200.engine import Engine
    eng = Engine()
    eng.set_track(ellipse)
    poses, _ = synth.random_poses(ellipse, 100000, np.random.default_rng(1002))
    poses = np.ascontiguousarray(poses[:, :3])
    r = eng.pure_pursuit_batch(poses, 0.8)
    perm = np.random.default_rng(1).permutation(100000)
    rp = eng.pure_pursuit_batch(poses[perm], 0.8)
    assert np.array_equal(rp.nearest_i, r.nearest_i[perm])
    assert np.array_equal(rp.actuation, r.actuation[perm])
    part = eng.pure_pursuit_batch(poses[40000:40100], 0.8)
    assert np.array_equal(part.nearest, r.nearest[40000:40100])
    assert (r.status > 0).all()
