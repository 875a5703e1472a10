"""Synthetic inputs for benchmarks and tests (SURVEY.md 8d): ellipse raceline, corridor
occupancy grid, randomised poses and opponents.  Host-side numpy; input generation only.
"""
import numpy as np

CAR_LENGTH = 0.58  # reference control/kinematic_mpc/kinematic_mpc.py:60
CAR_WIDTH = 0.31   # :61


def ellipse_track(n=2000, a=80.0, b=40.0, speed=8.0):
    """[n,5] float64 (x, y, v, psi, kappa); uniform in the ellipse parameter, endpoint excluded,
    psi = forward-difference tangent in [0, 2pi), counter-clockwise."""
    phi = 2.0 * np.pi * np.arange(n) / n
    x = a * np.cos(phi)
    y = b * np.sin(phi)
    dx = np.roll(x, -1) - x
    dy = np.roll(y, -1) - y
    psi = np.mod(np.arctan2(dy, dx), 2.0 * np.pi)
    kappa = a * b / (a * a * np.sin(phi) ** 2 + b * b * np.cos(phi) ** 2) ** 1.5
    return np.stack([x, y, np.full(n, speed), psi, kappa], axis=1)


def corridor_grid(a=80.0, b=40.0, half_width=1.5, res=0.05, margin=5.0):
    """uint8 occupancy [H,W] (0 free / 1 occupied), origin (-a-margin, -b-margin); a cell is free
    when the first-order distance of its centre to the ellipse is <= half_width."""
    ox, oy = -a - margin, -b - margin
    w = int(round(2 * (a + margin) / res))
    h = int(round(2 * (b + margin) / res))
    xs = ox + (np.arange(w) + 0.5) * res
    occ = np.empty((h, w), dtype=np.uint8)
    for r0 in range(0, h, 256):  # row blocks keep the temporaries small
        ys = oy + (np.arange(r0, min(r0 + 256, h)) + 0.5) * res
        X, Y = np.meshgrid(xs, ys)
        rr = np.sqrt((X / a) ** 2 + (Y / b) ** 2)
        grad = np.sqrt((X / (a * a)) ** 2 + (Y / (b * b)) ** 2) / np.maximum(rr, 1e-12)
        dist = np.abs(rr - 1.0) / np.maximum(grad, 1e-12)
        occ[r0:r0 + ys.shape[0]] = (dist > half_width).astype(np.uint8)
    return occ, (ox, oy), res


def _arc(track):
    seg = np.hypot(np.diff(track[:, 0], append=track[0, 0]), np.diff(track[:, 1], append=track[0, 1]))
    return np.concatenate([[0.0], np.cumsum(seg)])  # [n+1], last = perimeter


def random_poses(track, s, rng):
    """[s,4] (x, y, theta, velocity) scattered around the raceline."""
    n = track.shape[0]
    idx = rng.integers(0, n, size=s)
    lat = np.clip(rng.normal(0.0, 0.3, size=s), -1.0, 1.0)
    psi = track[idx, 3]
    x = track[idx, 0] - lat * np.sin(psi)
    y = track[idx, 1] + lat * np.cos(psi)
    th = psi + rng.normal(0.0, 0.1, size=s)
    v = rng.uniform(2.0, 8.0, size=s)
    return np.stack([x, y, th, v], axis=1), idx


def random_opponents(track, idx, k, rng):
    """[s,k,3] map-frame (x, y, theta), 1..5 m ahead of each pose's waypoint along the raceline
    (SURVEY 8d suggested 0.5..3 m, which puts an opponent inside the ego footprint at t=0 in most
    8-opponent scenarios and makes every candidate collide)."""
    n = track.shape[0]
    s = idx.shape[0]
    arc = _arc(track)
    ahead = rng.uniform(1.0, 5.0, size=(s, k))
    target = np.mod(arc[idx][:, None] + ahead, arc[-1])
    j = np.clip(np.searchsorted(arc, target, side="right") - 1, 0, n - 1)
    lat = rng.normal(0.0, 0.4, size=(s, k))
    psi = track[j, 3]
    x = track[j, 0] - lat * np.sin(psi)
    y = track[j, 1] + lat * np.cos(psi)
    th = psi + rng.normal(0.0, 0.1, size=(s, k))
    return np.stack([x, y, th], axis=2)


def opponent_velocities(track, opp, rng, lo=2.0, hi=8.0):
    """[..., 2] map-frame velocities (vx, vy) of opponents `opp` [..., 3]: a speed drawn from
    U(lo, hi) m/s along each opponent's heading.  (`track` is taken for symmetry with the other
    scenario builders.)"""
    opp = np.asarray(opp, dtype=np.float64)
    v = rng.uniform(lo, hi, size=opp.shape[:-1])
    return np.stack([v * np.cos(opp[..., 2]), v * np.sin(opp[..., 2])], axis=-1)


def scenario_batch(track, s, k, seed):
    rng = np.random.default_rng(seed)
    poses, idx = random_poses(track, s, rng)
    opp = random_opponents(track, idx, k, rng)
    n_opp = rng.integers(1, k + 1, size=s).astype(np.int32) if k > 0 else np.zeros(s, np.int32)
    return poses, opp, n_opp


DEFAULT_LOOKAHEADS = np.array([0.4, 0.6, 0.8, 1.0])  # lattice_planner.py:228
DEFAULT_WIDTHS = np.linspace(-1.0, 1.0, num=7)       # lattice_planner.py:229


def goal_grid(config):
    """(lookaheads, widths) of the BASELINE configs: 1/4 -> 4x7, 3 -> 64x64, 5 -> 256x256."""
    if config in (1, 4):
        return DEFAULT_LOOKAHEADS.copy(), DEFAULT_WIDTHS.copy()
    if config == 3:
        return np.linspace(0.5, 4.0, 64), np.linspace(-1.2, 1.2, 64)
    if config == 5:
        return np.linspace(0.5, 4.0, 256), np.linspace(-1.2, 1.2, 256)
    raise ValueError(config)
