"""Pins the CPU oracle to the reference: golden vectors minted by tests/golden/make_golden.py from
the UNMODIFIED reference functions (utils/utils.py, pure_pursuit.py) and the SURVEY appendix-C
known answers."""
import os

import numpy as np

from oracle import c_oracle as co


def _check_pp(g, wp):
    o = co.pure_pursuit_batch(wp, g["poses"], float(g["lookahead_distance"]))
    assert np.array_equal(o["nearest_i"], g["nearest_i"])          # bit-exact indices
    np.testing.assert_allclose(o["nearest"], g["nearest"], rtol=0, atol=1e-12)
    m = g["nearest"][:, 2] < float(g["lookahead_distance"])         # intersect branch taken
    assert np.array_equal(o["lookahead_i"][m], g["lookahead_i"][m])
    assert np.array_equal(o["lookahead"][m, 3], g["lookahead"][m, 3])
    np.testing.assert_allclose(o["lookahead"][m, :3], g["lookahead"][m, :3], rtol=0, atol=1e-9)
    np.testing.assert_allclose(o["actuation"], g["actuation"], rtol=0, atol=1e-12)


def test_pure_pursuit_spielberg(golden_spielberg):
    _check_pp(golden_spielberg, golden_spielberg["waypoints"])


def test_pure_pursuit_ellipse(golden_ellipse, ellipse):
    _check_pp(golden_ellipse, ellipse)


def test_survey_appendix_c_known_answers(golden_spielberg):
    wp = golden_spielberg["waypoints"]
    xy = wp[:, :2]
    p, d, t, i = co.nearest_point([0.0, -0.84], xy)
    assert i == 1690
    np.testing.assert_allclose([p[0], p[1], d, t], [-6.623233363824144e-04, -8.375283214769740e-01,
                                                    0.0025588800134247534, 0.7752037243334408],
                               rtol=1e-12)
    ip, i2, t2 = co.intersect_point([0.0, -0.84], 0.8, xy, i + t, wrap=True)
    assert i2 == 3   # found in the wrap loop (seam crossing)
    np.testing.assert_allclose([ip[0], ip[1], t2], [-0.7733906818796472, -1.0446139124833267,
                                                    0.7760054648027157], rtol=1e-10)
    assert co.intersect_point([5.0, 5.0], 0.8, xy, 1659.0651423516027651, wrap=True) == (None, None, None)
    sp, st = co.get_actuation(0.3, [1.0, 0.5, 4.0], [0.2, 0.1], 0.8, 0.33)
    assert sp == 4.0
    np.testing.assert_allclose(st, 0.1491560800289004, rtol=1e-13)
    o = co.pure_pursuit_batch(wp, [[0.0, -0.84, 3.40], [-20.0, -6.0, 3.4], [5.0, 5.0, 0.0]], 0.8)
    np.testing.assert_allclose(o["actuation"][:, 0], [-0.00035935558090650324, 0.22560092622792158,
                                                      -1.3435444691165728], rtol=1e-10)
    assert o["status"].tolist() == [1, 1, 2]


def test_intersect_point_variants(golden_spielberg, golden_misc):
    xy, m = golden_spielberg["waypoints"][:, :2], golden_misc
    for k in range(m["ip_t"].shape[0]):
        p, i, t = co.intersect_point(m["ip_points"][k], m["ip_radius"][k], xy, m["ip_t"][k],
                                     bool(m["ip_wrap"][k]))
        if m["ip_out"][k, 3] == 0:
            assert p is None
        else:
            assert i == m["ip_i"][k]
            np.testing.assert_allclose([p[0], p[1], t], m["ip_out"][k, :3], rtol=0, atol=1e-9)


def test_get_actuation_vectors(golden_misc):
    m = golden_misc
    for r, ref in zip(m["act_in"], m["act_out"]):
        out = co.get_actuation(r[0], r[1:4], r[4:6], r[6], 0.33)
        np.testing.assert_allclose(out, ref, rtol=0, atol=1e-14)


def test_argmin_and_length_cost_semantics(golden_misc):
    assert int(golden_misc["select"][0]) == 1                 # LatticePlanner.select([3,1,1,2])
    assert golden_misc["length_cost"].tolist() == [0.5, 0.25]  # get_length_cost
    assert int(np.argmin([3.0, 1.0, 1.0, 2.0])) == 1


def test_front_axle_errors_match_stanley_and_lqr(golden_spielberg):
    """StanleyPlanner.calc_theta_and_ef / controller / plan (stanley.py:57-139) and
    LQRPlanner.calc_control_points (lqr.py:60-102)"""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "stanley.npz"))
    front, idx = co.front_axle_batch(golden_spielberg["waypoints"], g["states"],
                                     float(g["wheelbase"]), float(g["k_path"]))
    assert np.array_equal(idx, g["target_index"])
    np.testing.assert_allclose(front, g["front"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(front[:, [5, 4]], g["plan"], rtol=0, atol=1e-12)
