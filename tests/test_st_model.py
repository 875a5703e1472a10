"""The numpy restatement of the single-track model (tests/st_model.py), pinned to numerics that do
not share its code: scipy's DOP853 on the equations as f1tenth_gym writes them, the linear fixed
point and closed-form steady state of the (yaw rate, slip) equations, and the kinematic bicycle
below v_kin.  The GPU tests compare the kernel against this restatement."""
import math

import numpy as np
from scipy.integrate import solve_ivp

from tests import st_model as st

P = st.DEFAULTS
L = P["lf"] + P["lr"]


def _gym_f(q, sv, a):
    """f1tenth_gym's vehicle_dynamics_st, written term by term from its source form"""
    x, y, d, v, psi, r, b = q
    mu, Cf, Cr, lf, lr, h, m, I = (P[k] for k in ("mu", "C_Sf", "C_Sr", "lf", "lr", "h", "m", "I"))
    g = 9.81
    if abs(v) < P["v_kin"]:
        return [v * math.cos(psi), v * math.sin(psi), sv, a, v / L * math.tan(d),
                a / L * math.tan(d) + v / (L * math.cos(d) ** 2) * sv, 0.0]
    return [v * math.cos(psi + b), v * math.sin(psi + b), sv, a, r,
            -mu * m / (v * I * L) * (lf ** 2 * Cf * (g * lr - a * h) + lr ** 2 * Cr * (g * lf + a * h)) * r
            + mu * m / (I * L) * (lr * Cr * (g * lf + a * h) - lf * Cf * (g * lr - a * h)) * b
            + mu * m / (I * L) * lf * Cf * (g * lr - a * h) * d,
            (mu / (v ** 2 * L) * (Cr * (g * lf + a * h) * lr - Cf * (g * lr - a * h) * lf) - 1) * r
            - mu / (v * L) * (Cr * (g * lf + a * h) + Cf * (g * lr - a * h)) * b
            + mu / (v * L) * Cf * (g * lr - a * h) * d]


def _run(q, sv, a, dt, n):
    q = tuple(np.array([c], np.float64) for c in q)
    for _ in range(n):
        q = st.rk4(q, sv, a, dt)
    return np.array([c[0] for c in q])


def test_rk4_against_dop853_in_the_dynamic_branch():
    q0 = [0.0, 0.0, 0.0, 3.0, 0.0, 0.0, 0.0]
    sv, a = 0.8, 2.0
    got = _run(q0, sv, a, 0.01, 50)
    ref = solve_ivp(lambda t, y: _gym_f(y, sv, a), (0.0, 0.5), q0, method="DOP853", rtol=1e-12, atol=1e-12)
    assert np.abs(got - ref.y[:, -1]).max() < 5e-6
    assert got[3] > P["v_kin"] and abs(got[6]) > 1e-3   # stayed dynamic, and slipped


def test_steady_state_cornering():
    v, d = 5.0, 0.1
    got = _run([0.0, 0.0, d, v, 0.0, 0.0, 0.0], 0.0, 0.0, 0.01, 300)
    mu, Cf, Cr, lf, lr, m, I = (P[k] for k in ("mu", "C_Sf", "C_Sr", "lf", "lr", "m", "I"))
    g = 9.81
    A = np.array([[-mu * m / (v * I * L) * (lf ** 2 * Cf * g * lr + lr ** 2 * Cr * g * lf),
                   mu * m / (I * L) * (lr * Cr * g * lf - lf * Cf * g * lr)],
                  [mu / (v ** 2 * L) * (Cr * g * lf * lr - Cf * g * lr * lf) - 1,
                   -mu / (v * L) * (Cr * g * lf + Cf * g * lr)]])
    rhs = -np.array([mu * m / (I * L) * lf * Cf * g * lr * d, mu / (v * L) * Cf * g * lr * d])
    r_ss, b_ss = np.linalg.solve(A, rhs)
    K = (1.0 / mu) * (1.0 / Cf - 1.0 / Cr)
    assert abs(got[5] - r_ss) < 1e-9 and abs(got[6] - b_ss) < 1e-9
    assert abs(got[5] - v * d / (L + K * v * v / g)) < 1e-9
    assert abs(got[5] - 1.2503978899636) < 1e-9 and abs(got[6] + 0.0684827384314) < 1e-9
    assert got[5] < 0.85 * v * math.tan(d) / L   # the kinematic bicycle turns 21 % faster


def test_kinematic_form_below_v_kin():
    # at v < v_kin with delta and v held, the step is the rear-axle kinematic bicycle with L = lf + lr
    v, d, dt = 0.3, 0.2, 0.01
    got = _run([1.0, -2.0, d, v, 0.4, 0.0, 0.0], 0.0, 0.0, dt, 100)
    w = v * math.tan(d) / L
    psi = 0.4 + w * 1.0
    x = 1.0 + v / w * (math.sin(psi) - math.sin(0.4))
    y = -2.0 - v / w * (math.cos(psi) - math.cos(0.4))
    assert abs(got[4] - psi) < 1e-12
    assert abs(got[0] - x) < 1e-10 and abs(got[1] - y) < 1e-10
    assert got[6] == 0.0
    # with sv and a held the yaw rate state follows d/dt (v tan(delta) / L)
    sv, a = 0.5, 1.0
    got = _run([0.0, 0.0, 0.0, 0.1, 0.0, 0.0, 0.0], sv, a, dt, 20)
    assert got[3] < P["v_kin"]
    assert abs(got[5] - got[3] * math.tan(got[2]) / L) < 1e-9


def test_mirror_symmetry():
    rng = np.random.default_rng(7)
    S = 64
    X = np.stack([rng.normal(0, 3, S), rng.normal(0, 3, S), rng.normal(0, 1, S), rng.uniform(0, 9, S)], axis=1)
    D = np.stack([rng.uniform(-0.4, 0.4, S), rng.normal(0, 1, S), rng.normal(0, 0.1, S)], axis=1)
    steer, target = rng.uniform(-0.4189, 0.4189, S), rng.uniform(0, 9, S)
    Xa, Da = X.copy(), D.copy()
    Xb = X * [1, -1, -1, 1]
    Db = -D
    for _ in range(5):
        Xa, Da = st.substep(Xa, Da, steer, target, 0.01, 9.51)
        Xb, Db = st.substep(Xb, Db, -steer, target, 0.01, 9.51)
    assert np.array_equal(Xb, Xa * [1, -1, -1, 1])
    assert np.array_equal(Db, -Da)
    assert (np.abs(X[:, 3]) < P["v_kin"]).any() and (X[:, 3] > P["v_switch"]).any()


def test_controls_follow_the_limits():
    d = np.array([0.0, 0.0, 0.3])
    v = np.array([2.0, 8.0, 8.0])
    sv, a = st.controls(d, v, np.array([0.4, -0.01, 0.3]), np.array([9.0, 20.0, 0.0]), 0.01, 9.51)
    assert np.allclose(sv, [3.2, -1.0, 0.0])
    assert np.allclose(a, [9.51, 9.51 * 7.319 / 8.0, -9.51])
