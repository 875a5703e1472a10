"""Moving opponents without a device: the new entry points' argument checks, the MOTION_FIELDS row,
and the reference for moving opponents on closed-form cases (tests/motion_oracle.py: plan_motion,
the float64 truth the GPU tests hold the kernel to, and collide_f32_motion, the float32 mirror)."""
import ctypes as C
import math

import numpy as np
import pytest

from f1tenth_planning_b200 import _lib, synth
from f1tenth_planning_b200.engine import _motion_array
from oracle import c_oracle as co
from tests import motion_oracle as MO

INVALID = -1
DIMS = dict(S=3, K=2, C=5, M=7)


def test_null_handle_rejected_by_every_new_entry_point():
    L = _lib.lib()
    pose = (C.c_double * 4)(0, 0, 0, 1)
    res = _lib.PlanResult()
    b = _lib.BatchCall(n_scenarios=1, max_opp=0, poses=C.addressof(pose))
    rc = _lib.RolloutConfig()
    assert L.f1l_default_rollout_config(C.byref(rc)) == 0
    fl = _lib.FleetBuffers()
    out = (C.c_float * 33)()
    assert L.f1l_plan_motion(None, C.addressof(pose), None, None, 0, 1.0, 0, C.byref(res)) == INVALID
    assert L.f1l_plan_batch_motion(None, C.byref(b), None, 1.0) == INVALID
    assert L.f1l_plan_batch_motion_dev(None, C.byref(b), None, 1.0, None) == INVALID
    assert L.f1l_rollout_predict_dev(None, C.byref(rc), None, C.byref(fl), None, None, 1.0, 4, 1, None,
                                     None, None) == INVALID
    assert L.f1l_debug_motion_ctx(None, out, 33) == INVALID


def test_motion_row_rejects_bad_host_arrays():
    row = _lib.MOTION_FIELDS["opp_vel"]
    assert row == (("float64",), ("S", "K", 2), _lib.IN)
    shape = _lib.shape_of(row, DIMS)
    good = np.zeros(shape)
    _lib.check_array("opp_vel", good, shape, row[0], "host")
    strided = np.zeros(shape[:-1] + (4,))[..., ::2]
    for bad in (good.astype(np.float32), np.zeros((4, 2, 2)), np.zeros((3, 2, 3)), good[None], strided,
                good.tolist()):
        with pytest.raises(ValueError):
            _lib.check_array("opp_vel", bad, shape, row[0], "host")
    # the engine's host path converts a float array to float64, but not a wrong shape
    assert _motion_array(good.astype(np.float32), "host", DIMS).dtype == np.float64
    with pytest.raises(ValueError):
        _motion_array(np.zeros((3, 3, 2)), "host", DIMS)


def test_synth_opponent_velocities_follow_heading():
    track = synth.ellipse_track()
    poses, opp, n_opp = synth.scenario_batch(track, 50, 4, 7)
    v = synth.opponent_velocities(track, opp, np.random.default_rng(1), 2.0, 8.0)
    assert v.shape == opp.shape[:2] + (2,)
    speed = np.hypot(v[..., 0], v[..., 1])
    assert (speed >= 2.0).all() and (speed <= 8.0).all()
    np.testing.assert_allclose(np.arctan2(v[..., 1], v[..., 0]), np.angle(np.exp(1j * opp[..., 2])), atol=1e-12)
    # a scenario batch draws exactly as before: the velocities come from their own generator
    p2, o2, n2 = synth.scenario_batch(track, 50, 4, 7)
    assert np.array_equal(p2, poses) and np.array_equal(o2, opp) and np.array_equal(n2, n_opp)


# ---- the oracle ---------------------------------------------------------------------------------
def _straight(n=1001):
    x = np.linspace(-50.0, 50.0, n)
    return np.stack([x, np.zeros(n), np.full(n, 8.0), np.zeros(n), np.zeros(n)], axis=1)


@pytest.fixture(scope="module")
def straight():
    """one straight candidate of length 3 m along +x from the origin (heading 0)"""
    cfg = co.default_config()
    world = co.World_(_straight(), np.array([3.0]), np.array([0.0]))
    return cfg, world


def _ego_x(cfg, world, pose):
    o = co.plan(cfg, world, pose, None, want_states=True)
    assert o["flags"][0] & co.FLAG_VALID
    return o["states"][0, :, 0], o["params"][0, 2]


def _hits(cfg, world, pose, opp, vel, v_min=1.0):
    o = MO.plan_motion(cfg, world, pose, np.atleast_2d(opp), np.atleast_2d(vel), v_min)
    return bool(o["flags"][0] & co.FLAG_COLLIDE_OPP), o


def test_zero_velocities_equal_static_plan():
    track = synth.ellipse_track()
    la, wd = synth.goal_grid(4)
    occ, origin, res = synth.corridor_grid()
    world = co.World_(track, la, wd, grid=occ, grid_origin=origin, grid_res=res)
    cfg = co.default_config(kappa_max=3.0)
    n_hit = 0
    for seed in range(6):
        poses, opp, n_opp = synth.scenario_batch(track, 1, 6, seed)
        o = co.plan(cfg, world, poses[0], opp[0], want_states=True)
        m = MO.plan_motion(cfg, world, poses[0], opp[0], np.zeros((6, 2)), 1.0, want_states=True)
        for key in ("costs", "terms", "flags", "params", "goals", "states", "margins"):
            assert np.array_equal(o[key], m[key], equal_nan=True), key
        for key in ("best_idx", "best_cost", "no_feasible"):
            assert o[key] == m[key], key
        n_hit += int((o["flags"] & co.FLAG_COLLIDE_OPP).astype(bool).sum())
    assert n_hit > 0
    b = co.plan_batch(cfg, world, *synth.scenario_batch(track, 20, 4, 3)[:2],
                      n_opp=synth.scenario_batch(track, 20, 4, 3)[2])
    poses, opp, n_opp = synth.scenario_batch(track, 20, 4, 3)
    bm = MO.plan_batch_motion(cfg, world, poses, opp, np.zeros(opp.shape[:2] + (2,)), n_opp)
    for key in ("best_idx", "best_cost", "costs", "flags"):
        assert np.array_equal(b[key], bm[key], equal_nan=True), key


def test_head_on_collides_when_centres_reach_contact(straight):
    """Opponent ahead at D heading at the ego with speed u: at sample i the centres are
    d_i = D - x_i - u t_i apart, t_i = i s_f / ((M-1) v_e).  Aligned equal rectangles overlap iff
    |d_i| < car_length."""
    cfg, world = straight
    pose = np.array([0.0, 0.0, 0.0, 2.0])
    x, sf = _ego_x(cfg, world, pose)
    M = cfg.n_samples
    t = np.arange(M) * sf / ((M - 1) * 2.0)
    seen = set()
    for D in (2.0, 4.0, 6.0, 7.0, 7.5, 8.0, 8.3, 9.0, 11.0):
        for u in (0.0, 1.0, 3.0):
            d = D - x - u * t
            margin = np.abs(np.abs(d) - cfg.car_length).min()
            if margin < 1e-6:
                continue
            want = bool((np.abs(d) < cfg.car_length).any())
            got, _ = _hits(cfg, world, pose, [D, 0.0, math.pi], [-u, 0.0])
            assert got == want, (D, u)
            seen.add((want, u > 0))
    assert {(True, True), (False, True), (True, False), (False, False)} <= seen
    # the prediction matters: 7 m ahead is clear when parked, a collision at 3 m/s
    assert not _hits(cfg, world, pose, [7.0, 0.0, math.pi], [0.0, 0.0])[0]
    assert _hits(cfg, world, pose, [7.0, 0.0, math.pi], [-3.0, 0.0])[0]


def test_leader_moving_away_never_collides(straight):
    cfg, world = straight
    for v in (0.0, 0.5, 2.0, 4.0):        # v_e = max(v, v_min = 1)
        v_e = max(v, 1.0)
        pose = np.array([0.0, 0.0, 0.0, v])
        assert _hits(cfg, world, pose, [1.0, 0.0, 0.0], [0.0, 0.0])[0]
        for u in (v_e, 1.5 * v_e):
            assert not _hits(cfg, world, pose, [1.0, 0.0, 0.0], [u, 0.0])[0], (v, u)
    # v_min times a car at rest: timed at 1 m/s it catches a leader at 0.5 m/s, timed at 0.4 not
    pose = np.array([0.0, 0.0, 0.0, 0.0])
    assert _hits(cfg, world, pose, [1.0, 0.0, 0.0], [0.5, 0.0], v_min=1.0)[0]
    assert not _hits(cfg, world, pose, [1.0, 0.0, 0.0], [0.5, 0.0], v_min=0.4)[0]


def test_crossing_collides_only_when_arriving_with_the_ego(straight):
    """An opponent crossing the ego's line at x_c (heading +y, speed u) from y0 < 0 is on the line
    at t = -y0 / u; the ego is there at x_c / v_e."""
    cfg, world = straight
    pose = np.array([0.0, 0.0, 0.0, 2.0])
    xc, u = 2.0, 3.0
    y0 = -u * xc / 2.0
    assert _hits(cfg, world, pose, [xc, y0, math.pi / 2], [0.0, u])[0]
    assert not _hits(cfg, world, pose, [xc, y0, math.pi / 2], [0.0, 0.0])[0]   # parked: far off the line
    for early in (-1.0, 1.0):        # a second early or late: clear
        assert not _hits(cfg, world, pose, [xc, y0 + early * u, math.pi / 2], [0.0, u])[0]


def test_f32_mirror_agrees_with_f64_truth_away_from_margin():
    track = synth.ellipse_track()
    la, wd = synth.goal_grid(3)
    world = co.World_(track, la, wd)
    cfg = co.default_config(kappa_max=3.0)
    rng = np.random.default_rng(4)
    hl, hw = 0.5 * cfg.car_length, 0.5 * cfg.car_width
    rc2 = 4.0 * (hl * hl + hw * hw)
    n_cmp, n_hit, n_diff = 0, 0, 0
    for seed in range(4):
        pose, opp = synth.scenario_batch(track, 1, 6, seed)[:2]
        pose, opp = pose[0], opp[0]
        vel = synth.opponent_velocities(track, opp, rng, 2.0, 8.0) * rng.choice([-1.0, 1.0], size=(6, 1))
        o = MO.plan_motion(cfg, world, pose, opp, vel, 1.0, want_states=True)
        c, s = math.cos(pose[2]), math.sin(pose[2])
        dx, dy = opp[:, 0] - pose[0], opp[:, 1] - pose[1]
        loc = np.zeros((16, 4), np.float32)
        loc[:6] = np.stack([c * dx + s * dy, -s * dx + c * dy, np.cos(opp[:, 2] - pose[2]),
                            np.sin(opp[:, 2] - pose[2])], axis=1)
        wl = np.zeros((16, 2), np.float32)
        wl[:6] = np.stack([c * vel[:, 0] + s * vel[:, 1], -s * vel[:, 0] + c * vel[:, 1]], axis=1)
        k_t = np.float32(1.0 / ((cfg.n_samples - 1) * max(pose[3], 1.0)))
        valid = (o["flags"] & co.FLAG_VALID) != 0
        sv = o["states"][valid]
        hd = np.stack([np.cos(sv[..., 2]), np.sin(sv[..., 2])], axis=-1)
        mirror = np.zeros_like(o["flags"])
        mirror[valid] = MO.collide_f32_motion(sv, hd, o["params"][valid], loc, wl, k_t, 6,
                                              np.zeros(6, np.float32), np.zeros(2, np.int32), None, hl, hw, rc2)
        far = valid & (o["margins"][:, 0] > 1e-3)
        n_cmp += int(far.sum())
        n_hit += int((o["flags"][far] & co.FLAG_COLLIDE_OPP).astype(bool).sum())
        n_diff += int((mirror[far] & 2 != o["flags"][far] & 2).sum())
    assert n_cmp > 2000 and n_hit > 50
    assert n_diff == 0
