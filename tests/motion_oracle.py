"""The reference for planning against moving opponents, restated over the CPU oracle.

Opponent k, at opp[k] = (x, y, theta), moves at the constant map-frame velocity opp_vel[k] and keeps
its heading.  The ego, timed at v_e = max(pose[3], v_min), reaches sample i of a candidate of length
s_f at t_i = i s_f / ((M - 1) v_e); the opponent's footprint is then centred at
opp[k] + opp_vel[k] t_i.  Nothing else of a plan depends on the opponents, so:

- plan_motion is the oracle's float64 plan without opponents (trajectories, validity, map flags,
  cost terms) with the opponent test of oracle/c/f1o.c (sat_separation, the broad phase, the
  opponent margin) applied at the predicted centres, operation for operation in float64.  With
  every velocity zero its flags, margins, costs and argmin are those of c_oracle.plan with the
  opponents, bit for bit (tests/test_motion_abi.py).  It does not run the tracker.
- collide_f32_motion is the float32 mirror of the device predicate: eval_kernel's explicitly
  rounded operations (dt = s_f k_t, t_i = (float)i dt, centre (ox + wx t_i, oy + wy t_i), then the
  circle test and sat_collide), each one a separately rounded numpy float32 operation, on the
  device's own states, parameters and motion constants (Engine.debug_motion_ctx).  The map flags
  come from c_oracle.collide_f32.
"""
import math

import numpy as np

from oracle import c_oracle as co


def _cos_sin(a):
    """libm's cos / sin element by element, as the C oracle calls them"""
    a = np.asarray(a, dtype=np.float64)
    flat = a.ravel()
    return (np.array([math.cos(v) for v in flat]).reshape(a.shape),
            np.array([math.sin(v) for v in flat]).reshape(a.shape))


def _sat_separation(tx, ty, ca, sa, cb, sb, hl, hw):
    """f1o.c sat_separation: < 0 iff the two rectangles overlap"""
    c = np.abs(ca * cb + sa * sb)
    s = np.abs(sa * cb - ca * sb)
    rl = hl + hl * c + hw * s
    rw = hw + hl * s + hw * c
    e0 = np.abs(tx * ca + ty * sa) - rl
    e1 = np.abs(-tx * sa + ty * ca) - rw
    e2 = np.abs(tx * cb + ty * sb) - rl
    e3 = np.abs(-tx * sb + ty * cb) - rw
    return np.maximum(np.maximum(np.maximum(e0, e1), e2), e3)


def plan_motion(cfg, world, pose, opp, opp_vel, v_min=1.0, want_states=False):
    """the goal-grid plan against opponents `opp` [K,3] moving at `opp_vel` [K,2] (map frame):
    dict with costs, terms, flags, params, goals, margins (opponent margins at the predicted
    positions), best_idx, best_cost, no_feasible (and states with want_states)"""
    pose = np.asarray(pose, dtype=np.float64)
    opp = np.zeros((0, 3)) if opp is None else np.asarray(opp, dtype=np.float64).reshape(-1, 3)
    vel = np.zeros((0, 2)) if opp_vel is None else np.asarray(opp_vel, dtype=np.float64).reshape(-1, 2)
    if vel.shape[0] != opp.shape[0]:
        raise ValueError("one velocity per opponent")
    if not (math.isfinite(v_min) and v_min > 0):
        raise ValueError("v_min must be finite and positive")
    o = co.plan(cfg, world, pose, None, want_states=True)
    M = cfg.n_samples
    v_e = pose[3] if pose[3] > v_min else v_min
    hl, hw = 0.5 * cfg.car_length, 0.5 * cfg.car_width
    rc2 = 4.0 * (hl * hl + hw * hw)
    ct, stn = math.cos(pose[2]), math.sin(pose[2])
    flags = o["flags"].copy()
    costs = o["costs"].copy()
    margins = o["margins"].copy()
    valid = np.nonzero(flags & co.FLAG_VALID)[0]
    if opp.shape[0] and valid.size:
        st = o["states"][valid]                                      # [V,M,4]
        x, y = st[:, :, 0], st[:, :, 1]
        X = pose[0] + ct * x - stn * y
        Y = pose[1] + stn * x + ct * y
        ca, sa = _cos_sin(st[:, :, 2] + pose[2])
        t = np.arange(M, dtype=np.float64)[None, :] * o["params"][valid, 2:3] / (float(M - 1) * v_e)
        cb, sb = _cos_sin(opp[:, 2])
        m_opp = np.full(valid.size, np.inf)
        hit = np.zeros(valid.size, bool)
        for k in range(opp.shape[0]):
            tx = (opp[k, 0] + vel[k, 0] * t) - X
            ty = (opp[k, 1] + vel[k, 1] * t) - Y
            sep = _sat_separation(tx, ty, ca, sa, cb[k], sb[k], hl, hw)
            m_opp = np.minimum(m_opp, np.abs(sep).min(axis=1))
            hit |= ((tx * tx + ty * ty <= rc2) & (sep < 0.0)).any(axis=1)
        margins[valid, 0] = m_opp
        flags[valid[hit]] |= co.FLAG_COLLIDE_OPP
        costs[valid[hit]] = np.inf
    finite = np.isfinite(costs)
    best = int(np.argmin(costs)) if finite.any() else 0
    out = dict(costs=costs, terms=o["terms"], flags=flags, params=o["params"], goals=o["goals"],
               margins=margins, best_idx=best, best_cost=float(costs[best]) if finite.any() else math.inf,
               no_feasible=not finite.any())
    if want_states:
        out["states"] = o["states"]
    return out


def plan_batch_motion(cfg, world, poses, opp, opp_vel, n_opp=None, v_min=1.0):
    """plan_motion per scenario: opp [S,K,3], opp_vel [S,K,2] -> best_idx [S], best_cost [S],
    costs [S,C], flags [S,C]"""
    poses = np.asarray(poses, dtype=np.float64).reshape(-1, 4)
    S, K = poses.shape[0], opp.shape[1]
    rows = []
    for s in range(S):
        k = K if n_opp is None else int(n_opp[s])
        rows.append(plan_motion(cfg, world, poses[s], opp[s, :k], opp_vel[s, :k], v_min))
    return dict(best_idx=np.array([r["best_idx"] for r in rows], np.int32),
                best_cost=np.array([r["best_cost"] for r in rows]),
                costs=np.stack([r["costs"] for r in rows]), flags=np.stack([r["flags"] for r in rows]))


def collide_f32_motion(states, headings, params, opp_local, vel_local, k_t, n_opp, grid_xf, grid_i0, grid,
                       half_l, half_w, rc2):
    """float32 mirror of eval_kernel's moving-opponent predicate on the device's own float32
    states [C,M,4], headings [C,M,2] (cos, sin), params [C,4] (s_f in column 2), vehicle-frame
    opponents [16,4] (x, y, cos, sin) and velocities [16,2], and k_t -> flags [C] (opponent bit 2,
    map bit 4)"""
    f32 = np.float32
    st = np.asarray(states, dtype=f32)
    hd = np.asarray(headings, dtype=f32)
    Cn, M = st.shape[0], st.shape[1]
    x, y, cs, sn = st[:, :, 0], st[:, :, 1], hd[:, :, 0], hd[:, :, 1]
    hl, hw, rc2 = f32(half_l), f32(half_w), f32(rc2)
    dt = np.asarray(params, dtype=f32)[:, 2:3] * f32(k_t)           # fm(s_f, k_t)
    t = np.arange(M, dtype=f32)[None, :] * dt                       # fm((float)i, dt)
    hit = np.zeros(Cn, bool)
    op = np.asarray(opp_local, dtype=f32)
    vl = np.asarray(vel_local, dtype=f32)
    for k in range(int(n_opp)):
        ox, oy, oc, os_ = op[k]
        tx = (ox + vl[k, 0] * t) - x                                # fs(fa(ox, fm(wx, t)), x)
        ty = (oy + vl[k, 1] * t) - y
        d2 = tx * tx + ty * ty
        cc = np.abs(cs * oc + sn * os_)
        ss = np.abs(sn * oc - cs * os_)
        rl = hl + (hl * cc + hw * ss)
        rw = hw + (hl * ss + hw * cc)
        e0 = np.abs(tx * cs + ty * sn)
        e1 = np.abs(ty * cs - tx * sn)
        e2 = np.abs(tx * oc + ty * os_)
        e3 = np.abs(ty * oc - tx * os_)
        hit |= ((d2 <= rc2) & (e0 < rl) & (e1 < rw) & (e2 < rl) & (e3 < rw)).any(axis=1)
    flags = co.collide_f32(st, hd, np.zeros((16, 4), f32), 0, grid_xf, grid_i0, grid, half_l, half_w, rc2)
    return flags | np.where(hit, co.FLAG_COLLIDE_OPP, 0).astype(np.uint8)
