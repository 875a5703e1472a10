"""Numpy restatement of the dynamic single-track model of f1l_rollout_st_dev (include/f1l.h), in
float64 and in the kernel's order of operations (f1l_rollout.cuh st_deriv / st_substep), vectorised
over cars.  The CPU tests pin it to independent numerics (solve_ivp, the linear fixed point, the
kinematic bicycle); the GPU tests compare the kernel against it step by step."""
import numpy as np

G = 9.81
DEFAULTS = dict(mu=1.0489, C_Sf=4.718, C_Sr=5.4562, lf=0.15875, lr=0.17145, h=0.074, m=3.74, I=0.04712,
                max_steer_vel=3.2, v_switch=7.319, v_kin=0.5)


def deriv(q, sv, acc, p=DEFAULTS):
    """d/dt of q = (x, y, delta, v, psi, yaw rate, beta), each an array [S], with (sv, acc) held"""
    _, _, d, v, psi, r, b = q
    L = p["lf"] + p["lr"]
    kr = (p["mu"] * p["m"]) / (p["I"] * L)
    kb = p["mu"] / L
    Ff = G * p["lr"] - acc * p["h"]
    Fr = G * p["lf"] + acc * p["h"]
    cf = p["C_Sf"] * Ff
    cr = p["C_Sr"] * Fr
    A1 = (p["lf"] * p["lf"]) * cf + (p["lr"] * p["lr"]) * cr
    A2 = p["lr"] * cr - p["lf"] * cf
    A3 = p["lf"] * cf
    B1 = cr + cf
    kin = np.abs(v) < p["v_kin"]
    with np.errstate(divide="ignore", invalid="ignore"):
        # kinematic form (|v| < v_kin)
        sd, cd = np.sin(d), np.cos(d)
        td = sd / cd
        k_dpsi = (v / L) * td
        k_dr = (acc / L) * td + (v / ((L * cd) * cd)) * sv
        # dynamic form
        iv = 1.0 / v
        d_dr = kr * ((A2 * b + A3 * d) - (A1 * iv) * r)
        d_db = ((((kb * A2) * iv) * iv) - 1.0) * r - (kb * iv) * (B1 * b - cf * d)
    ang = np.where(kin, psi, psi + b)
    return (v * np.cos(ang), v * np.sin(ang), np.broadcast_to(sv, v.shape), np.broadcast_to(acc, v.shape),
            np.where(kin, k_dpsi, r), np.where(kin, k_dr, d_dr), np.where(kin, 0.0, d_db))


def controls(d, v, steer, target, dt, max_accel, p=DEFAULTS):
    """(sv, acc) of one substep: steer already clamped to +-max_steer"""
    sv = np.minimum(np.maximum((steer - d) / dt, -p["max_steer_vel"]), p["max_steer_vel"])
    with np.errstate(divide="ignore", invalid="ignore"):
        a_pos = np.where(v > p["v_switch"], (max_accel * p["v_switch"]) / v, max_accel)
    acc = np.minimum(np.maximum((target - v) / dt, -max_accel), a_pos)
    return sv, acc


def rk4(q, sv, acc, dt, p=DEFAULTS):
    """one classical RK4 step of q (7 arrays) with (sv, acc) held"""
    q0 = [np.asarray(c, np.float64) for c in q]
    hdt, dt6 = 0.5 * dt, dt / 6.0
    k = deriv(q0, sv, acc, p)
    s = list(k)
    k = deriv([a + hdt * b for a, b in zip(q0, k)], sv, acc, p)
    s = [a + 2.0 * b for a, b in zip(s, k)]
    k = deriv([a + hdt * b for a, b in zip(q0, k)], sv, acc, p)
    s = [a + 2.0 * b for a, b in zip(s, k)]
    k = deriv([a + dt * b for a, b in zip(q0, k)], sv, acc, p)
    s = [a + b for a, b in zip(s, k)]
    return tuple(a + dt6 * b for a, b in zip(q0, s))


def substep(X, D, steer, target, dt, max_accel, p=DEFAULTS):
    """one substep of live cars: X [S,4] (x, y, psi, v), D [S,3] (delta, yaw rate, beta), steer
    clamped to +-max_steer, target speed -> (X, D) new arrays"""
    sv, acc = controls(D[:, 0], X[:, 3], steer, target, dt, max_accel, p)
    x, y, d, v, psi, r, b = rk4((X[:, 0], X[:, 1], D[:, 0], X[:, 3], X[:, 2], D[:, 1], D[:, 2]), sv, acc, dt, p)
    return np.stack([x, y, psi, v], axis=1), np.stack([d, r, b], axis=1)
