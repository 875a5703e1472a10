"""Every cost term of a single query (f1l_plan_result.terms) recomputed in float64 from the device's
own float32 trajectories: teacher-forced, so that the tolerance is the FP32 rounding of the kernel
rather than the oracle's 1e-4.

eval_kernel's raceline-deviation pass takes more shortcuts than any other loop of the library: a
float32 line form of every window segment built per scenario in the vehicle frame, samples and
table in units of EVAL_DEV_UNIT, a table padded to nseg_pad, two segments per trip, the odd last
sample row split over two lane halves that meet in one shuffle, the halving min / sqrt.approx
reduction and, in prune mode, a [k_begin, k_end) range from a chord-midpoint bound.  The window is
[seg0, seg0 + W) cyclic over the N - 1 open segments, seg0 = (i_ego - W // 4) mod (N - 1).  The
queries here sit where those shortcuts can go wrong: windows of 1 ... 129 segments and the whole
track, poses whose window wraps the seam on either side, a 2 cm raceline on which most samples lie
beyond the window's far end, 50 m segments far from the pose, zero-length segments, every sample
count edge of the instance table (smallest and largest M of each bucket, the split and unsplit odd
row), pruned and full scans, colliding candidates, both generators and the persistent wide grid.

References (numpy, float64; the per-term derivations of the bounds are in the docstrings of the
functions that form them).  test_reference_matches_nearest_point and
test_crafted_cases_reach_every_class need no GPU.
"""
import functools
import os

import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from oracle import c_oracle as co
from tests import helpers as H
from tests.test_eval_choice import eval_builds, eval_choice
from tests.test_gpu_intersect import tracks as intersect_tracks

gpu = pytest.mark.gpu

U = 2.0 ** -24           # unit roundoff of float32
EPS_SQRT = 2.0 ** -22    # relative error allowed sqrt.approx.ftz.f32 (PTX ISA: 2^-23, one more bit for
                         # the rounding of its result)
CHUNK = 1 << 21          # elements per [candidates, samples, segments] block of the reference
WINDOWS = (1, 2, 3, 31, 32, 33, 63, 64, 65, 128, 129)
LA = np.array([0.5, 1.5, 3.0, 6.0])    # goal rows; 6 m runs past the far end of short windows
WD = np.array([-0.8, 0.0, 0.8])
LATS = (0.0, 0.5, -0.5)                # lateral offsets of the crafted poses
EGO_CLASSES = ("0", "1", "W/4-1", "W/4", "N-3", "N-2")
SMALL = ("small3", "small9", "small33")
# goals (vehicle frame) whose trajectories run past the far end of a short window, and goals
# behind-left / behind-right of the car, around a hairpin
GOALS = np.array([[8.0, 0.0, 0.0], [12.0, 1.0, 0.2], [5.0, -2.0, -0.5], [1.5, 4.0, 2.8],
                  [1.5, -4.0, -2.8], [-1.0, 3.0, 3.0], [-1.0, -3.0, -3.0]])


# -- tracks -----------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def tracks():
    """test_gpu_intersect's tracks, Spielberg (golden file), and the ellipse with waypoint 0
    repeated at the front and waypoint 999 repeated mid-track: zero-length segments 0 and 1000,
    as real raceline files contain them"""
    out = dict(intersect_tracks())
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pp_spielberg.npz")
    out["spielberg"] = np.load(golden)["waypoints"]
    e = synth.ellipse_track()
    out["dup"] = e[np.concatenate([[0], np.arange(1000), [999], np.arange(1000, e.shape[0])])]
    return out


TRACKS = ("ellipse", "dense", "arc", "sparse", "small3", "small9", "small33", "offset", "spielberg", "dup")


def windows(name):
    n = tracks()[name].shape[0]
    w = set(WINDOWS)
    if name in SMALL:
        w |= {n - 2, n - 1, n, 0}
    return sorted(w)


# -- float64 references ---------------------------------------------------------------------------
def seg_dist(P, A, B):
    """distance [..., W] of the points P [..., 2] to the segments A[k] -> B[k] ([W, 2]) with
    nearest_point's clamp of t to [0, 1] (utils/utils.py:53-65); a zero-length segment's distance
    is the distance to its point"""
    D = B - A
    l2 = (D * D).sum(-1)
    dx = P[..., 0, None] - A[:, 0]
    dy = P[..., 1, None] - A[:, 1]
    t = np.clip((dx * D[:, 0] + dy * D[:, 1]) / np.where(l2 > 0.0, l2, 1.0), 0.0, 1.0)
    return np.hypot(dx - t * D[:, 0], dy - t * D[:, 1])


def nearest(track, p):
    """(distance [W], first minimum): the exhaustive search over every open segment"""
    xy = track[:, :2]
    d = seg_dist(np.asarray(p[:2], np.float64)[None], xy[:-1], xy[1:])[0]
    return d, int(np.argmin(d))


def window_rule(n_pts, window, i_ego):
    """(seg0, W) the sampler must set: W = N - 1 for window <= 0 or > N - 1"""
    nseg = n_pts - 1
    W = nseg if window <= 0 or window > nseg else window
    return (i_ego - W // 4) % nseg, W


def to_vehicle(xy, pose):
    """map-frame points -> the vehicle frame of the float64 pose"""
    c, s = np.cos(pose[2]), np.sin(pose[2])
    dx, dy = xy[..., 0] - pose[0], xy[..., 1] - pose[1]
    return np.stack([c * dx + s * dy, -s * dx + c * dy], axis=-1)


def gamma(n):
    return n * U / (1.0 - n * U)


def deviation_reference(states, track, pose, seg0, W):
    """(ref, lo, hi) [C]: the float64 raceline deviation of each candidate -- the mean over its M
    samples of the minimum distance to the window segments (seg0 + k) mod (N - 1), k < W -- and the
    interval the FP32 kernel's value must lie in.  The window is moved into the vehicle frame of the
    float64 pose; the samples are the device's float32 states, widened exactly.

    Per sample i and segment k (u = 2^-24; A, B the segment's vehicle-frame ends, s the sample, d
    the exact distance) the kernel's distance sqrt(d2'_ik) before the square root's own error is
    within
        e_ik = u (2 d + 10 |s| + 40 |A| + 20 |B|) + 1e-14 m
    of d_ik, to first order:
      - start A: fl32(p0 - pose), rotated by fl32(cos), fl32(sin) with one multiply and one FMA:
        each component within 4u |A|, the point within 6u |A|; the direction D = B - A likewise
        within 6u |D|;
      - unit vector and half length from rsqrtf (2 ulp = 4u) and the roundings of l2, ux, uy and
        l2 * il: |U'| = 1 +- 6u, its direction within 2u, h' = |D'| / 2 (1 +- 6u).  The line form
        so describes a segment whose ends lie within 6u |A| and 6u |A| + 14u |D| of A and B, and
        distance to a segment is 1-Lipschitz in its ends; |U'| != 1 scales the sample's offset
        from A by 1 +- 6u: 6u (|s| + |A|);
      - evaluation: T1.x (3 roundings) 3u (|A| + h), T1.y 2u |A|, q and n two FMAs each
        2u (|s| + |A| + h), the saturating add u (d + h), e^2 + n^2 u d: together
        u (4 |s| + 9 |A| + 6 h + 2 d);
    which sum to u (2 d + 10 |s| + 21 |A| + 17 |D|) <= the e_ik above with |D| <= |A| + |B|.  The
    1e-14 m covers flush-to-zero of squared distances below 2^-126 table units (~2e-15 m).
    The device's minimum over its k then lies in [lo_i, hi_i] with lo_i = max(0, min_k (d_ik -
    e_ik)) and hi_i = d_ik* + e_ik* (k* the exact argmin); sqrt.approx multiplies it by 1 +-
    EPS_SQRT; the M-term sum in any order and the scaling by (EVAL_DEV_UNIT * fl(1/M)) add at most
    gamma(M + 1) relative."""
    nseg = track.shape[0] - 1
    idx = (seg0 + np.arange(W)) % nseg
    A = to_vehicle(track[idx, :2], pose)
    B = to_vehicle(track[idx + 1, :2], pose)
    rA, rB = np.hypot(A[:, 0], A[:, 1]), np.hypot(B[:, 0], B[:, 1])
    C, M = states.shape[:2]
    S = states[..., :2].astype(np.float64)
    rs = np.hypot(S[..., 0], S[..., 1])
    ref, lo, hi = np.zeros(C), np.zeros(C), np.zeros(C)
    step = max(1, CHUNK // (M * W))
    for c0 in range(0, C, step):
        sl = slice(c0, c0 + step)
        d = seg_dist(S[sl], A, B)
        e = U * (2.0 * d + 10.0 * rs[sl, :, None] + 40.0 * rA + 20.0 * rB) + 1e-14
        k = d.argmin(-1)[..., None]
        dmin = np.take_along_axis(d, k, -1)[..., 0]
        ref[sl] = dmin.mean(-1)
        lo[sl] = np.maximum((d - e).min(-1), 0.0).sum(-1) / M
        hi[sl] = (dmin + np.take_along_axis(e, k, -1)[..., 0]).sum(-1) / M
    g = gamma(M + 1)
    return ref, lo * (1.0 - EPS_SQRT) * (1.0 - g), hi * (1.0 + EPS_SQRT) * (1.0 + g)


def _ratio(got, ref, bound):
    """max |got - ref| / bound (0 where both are zero)"""
    err = np.abs(np.asarray(got, np.float64) - ref)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0.0, 0.0, err / bound)
    return float(r.max()) if r.size else 0.0


def check_query(eng, track, pose, d, window, acc, prev=None):
    """every term of one single query against the float64 references; updates acc (max error /
    bound per term, class counts)"""
    cfg = eng.config
    M, n_shift, n_cull = int(cfg.n_samples), int(cfg.n_shift), int(cfg.n_cull)
    f, i = eng.debug_query_ctx()
    i_ego, seg0, W = int(i[2]), int(i[3]), int(i[4])
    n = track.shape[0]
    # the window
    assert (seg0, W) == window_rule(n, window, i_ego), (window, i_ego, seg0, W)
    dist, best = nearest(track, pose)
    assert abs(dist[i_ego] - dist[best]) <= 1e-12 * max(dist[best], 1.0), (i_ego, best, dist[i_ego], dist[best])
    if i_ego != best:
        acc["ego_tie"] = acc.get("ego_tie", 0) + 1
    acc["queries"] = acc.get("queries", 0) + 1
    acc.setdefault("windows", set()).add(W)
    nseg = n - 1
    for name, j in zip(EGO_CLASSES, (0, 1, (W // 4 - 1) % nseg, (W // 4) % nseg, n - 3, n - 2)):
        if i_ego == j:
            acc.setdefault("ego", {})[name] = acc.setdefault("ego", {}).get(name, 0) + 1
    if (seg0 + W > nseg) or seg0 == 0:
        acc["seam_windows"] = acc.get("seam_windows", 0) + 1
    # invalid candidates: every term 0
    valid = (d.flags & co.FLAG_VALID) != 0
    assert (d.terms[~valid] == 0.0).all(), np.nonzero(d.terms[~valid])[0][:5]
    acc["invalid"] = acc.get("invalid", 0) + int((~valid).sum())
    acc["valid"] = acc.get("valid", 0) + int(valid.sum())
    if not valid.any():
        return
    T = d.terms[valid]
    st = d.states[valid]
    # length: __fdividef(1, s_f), 2 ulp
    sf = d.params[valid, 2].astype(np.float64)
    ref = 1.0 / sf
    r = _ratio(T[:, 0], ref, 2.0 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64))
    _update(acc, "len", r)
    # max |kappa|: the same float32 maximum
    ak = np.abs(st[..., 3])
    assert np.array_equal(T[:, 1], ak.max(-1)), "max |kappa|"
    _update(acc, "max_kappa", 0.0)
    # mean |kappa|: an M-term float32 sum in any order, times fl(1/M): gamma(M + 1) relative
    ref = ak.astype(np.float64).mean(-1)
    _update(acc, "mean_kappa", _ratio(T[:, 2], ref, gamma(M + 1) * ref))
    # similarity: sum_{i < M - n_shift - n_cull} (theta_i - prev_{i + n_shift})^2; each difference
    # rounded once (2u on its square), the n FMAs and the warp sum in any order: gamma(n + 3)
    m = M - n_shift - n_cull
    if prev is None or m <= 0:
        assert (T[:, 3] == 0.0).all(), "similarity without a previous path / an empty range"
        _update(acc, "sim", 0.0)
    else:
        dd = st[:, :m, 2].astype(np.float64) - prev[n_shift:n_shift + m].astype(np.float64)
        ref = (dd * dd).sum(-1)
        _update(acc, "sim", _ratio(T[:, 3], ref, gamma(m + 3) * ref))
    # raceline deviation
    ref, lo, hi = deviation_reference(st, track, pose, seg0, W)
    got = T[:, 4].astype(np.float64)
    bound = np.where(got >= ref, hi - ref, ref - lo)
    r = _ratio(got, ref, bound)
    _update(acc, "dev", r)
    assert r <= 1.0, ("deviation", r, np.nonzero(np.abs(got - ref) > bound)[0][:5], got[:3], ref[:3])
    for k in ("len", "mean_kappa", "sim"):
        assert acc["max_ratio"][k] <= 1.0, (k, acc["max_ratio"][k])


def _update(acc, key, r):
    mr = acc.setdefault("max_ratio", {})
    mr[key] = max(mr.get(key, 0.0), r)


def _record(name, acc):
    out = dict(acc)
    if "windows" in out:
        out["windows"] = sorted(int(w) for w in out["windows"])
    if "shapes" in out:
        out["shapes"] = sorted(out["shapes"])
    H.record_parity("cost_terms_" + name, out)


# -- crafted cases ------------------------------------------------------------------------------
def ego_targets(n, W):
    nseg = n - 1
    return sorted({0, 1, (W // 4 - 1) % nseg, (W // 4) % nseg, n - 3, n - 2} & set(range(nseg)))


def ego_poses(track, W, rng):
    """poses [m, 4] at the midpoint of every target segment of window W, on the raceline and
    0.5 m to either side, heading along the segment"""
    xy = track[:, :2]
    nseg = xy.shape[0] - 1
    out = []
    for j in ego_targets(xy.shape[0], W):
        a, b = xy[j], xy[j + 1]
        k = j
        while np.hypot(*(xy[k + 1] - xy[k])) == 0.0:   # a zero-length segment: the next one's normal
            k = (k + 1) % nseg
        u = (xy[k + 1] - xy[k]) / np.hypot(*(xy[k + 1] - xy[k]))
        for lat in LATS:
            p = 0.5 * (a + b) + lat * np.array([-u[1], u[0]])
            out.append([p[0], p[1], np.arctan2(u[1], u[0]) + rng.normal(0.0, 0.05), rng.uniform(2.0, 8.0)])
    return np.array(out)


def ref_ego(track, p, name):
    """the reference's i_ego of pose p: co.nearest_point, except on the zero-length track, where
    nearest_point's NaN of 0 / 0 wins (np.argmin) and the exhaustive search above stands in"""
    if name == "dup":
        return nearest(track, p)[1]
    return co.nearest_point(p[:2], np.ascontiguousarray(track[:, :2]))[3]


def shape_ms():
    """[(row, [M...])]: per row of the instance table the smallest and largest M of its bucket,
    for odd S one M whose last sample row is split (M - (S - 1) SG <= SG / 2, with a sample in it)
    and one whose is not, and M = 2, 3 in the first row"""
    out, lo = [], 2
    for r in eval_builds():
        ms = {lo, r["m_max"]}
        if lo == 2:
            ms |= {2, 3}
        if r["s"] % 2:
            base = (r["s"] - 1) * r["sg"]
            ms |= {m for m in (base + 1, base + r["sg"] // 2, base + r["sg"] // 2 + 1) if lo <= m <= r["m_max"]}
        out.append((r, sorted(ms)))
        lo = r["m_max"] + 1
    return out


def split_odd(r, M):
    return r["s"] % 2 == 1 and M - (r["s"] - 1) * r["sg"] <= r["sg"] // 2


# -- no GPU ---------------------------------------------------------------------------------------
def test_reference_matches_nearest_point():
    """the numpy segment distance against co.nearest_point over the whole track (W = N - 1) on a
    few hundred points: distance within 1e-12 and the same segment"""
    rng = np.random.default_rng(17)
    worst = 0.0
    for name in ("ellipse", "sparse", "small9", "arc"):
        track = tracks()[name]
        xy = np.ascontiguousarray(track[:, :2])
        lo, hi = xy.min(0), xy.max(0)
        span = hi - lo
        P = rng.uniform(lo - 0.1 * span, hi + 0.1 * span, (100, 2))
        for p in P:
            d, k = nearest(track, p)
            _, od, _, oi = co.nearest_point(p, xy)
            assert abs(d[k] - od) <= 1e-12 * max(od, 1.0), (name, p, d[k], od)
            assert k == oi or abs(d[oi] - d[k]) <= 1e-12 * max(od, 1.0), (name, p, k, oi)
            worst = max(worst, abs(d[k] - od))
    # a zero-length segment: the distance to its point
    d = seg_dist(np.array([[3.0, 4.0]]), np.array([[0.0, 0.0]]), np.array([[0.0, 0.0]]))
    assert d[0, 0] == 5.0
    H.record_parity("cost_terms_reference_pin", {"points": 400, "max_abs_diff": worst})


def test_crafted_cases_reach_every_class():
    """the crafted poses reach every i_ego class on every track (by the reference's nearest
    point), and the sample counts reach the bucket edges and both odd-row cases of every row"""
    record = {}
    rng = np.random.default_rng(0)
    for name in TRACKS:
        track = tracks()[name]
        n = track.shape[0]
        got = {}
        for W in windows(name):
            _, Wr = window_rule(n, W, 0)
            for p in ego_poses(track, Wr, rng):
                j = ref_ego(track, p, name)
                for cls, t in zip(EGO_CLASSES, (0, 1, (Wr // 4 - 1) % (n - 1), (Wr // 4) % (n - 1), n - 3, n - 2)):
                    if j == t:
                        got[cls] = got.get(cls, 0) + 1
        record[name] = got
        for cls in EGO_CLASSES:
            assert got.get(cls, 0) > 0, (name, cls, got)
    rows = shape_ms()
    assert len(rows) == len(eval_builds())
    lo = 2
    for r, ms in rows:
        assert lo in ms and r["m_max"] in ms, (r, ms)
        if lo == 2:
            assert {2, 3} <= set(ms)
        if r["s"] % 2:
            both = [split_odd(r, m) for m in range(lo, r["m_max"] + 1)]
            if any(both):
                assert any(split_odd(r, m) and m > (r["s"] - 1) * r["sg"] for m in ms), (r, ms)
            if not all(both):
                assert any(not split_odd(r, m) for m in ms), (r, ms)
        record["M_%d" % r["m_max"]] = {"ms": ms, "split_odd": [m for m in ms if split_odd(r, m)]}
        lo = r["m_max"] + 1
    H.record_parity("cost_terms_crafted_classes", record)


# -- GPU ------------------------------------------------------------------------------------------
def _engine(track, **cfg):
    from f1tenth_planning_b200.engine import Engine
    cfg.setdefault("kappa_max", 0.0)
    eng = Engine(**cfg)
    eng.set_track(track)
    eng.set_goal_grid(LA, WD)
    eng.set_prev_path(None)
    eng.set_stats(True)
    return eng


def _plan(eng, track, pose, window, acc, prev=None, opp=None, goals=None):
    """one single query with the pruned and the full window scan, both checked; the deviation-pass
    counters checked on the way"""
    out = []
    for prune in (0, 1):
        eng.configure(prune_window=prune)
        eng.stats()
        if goals is None:
            d = eng.plan(pose, opp, update_prev=False, want_states=True)
        else:
            d = eng.plan_goals(pose, goals, opp, update_prev=False, want_states=True)
        steps, cands = eng.stats()
        check_query(eng, track, pose, d, window, acc, prev)
        W = int(eng.debug_query_ctx()[1][4])
        nseg_pad = (W + 31) & ~31
        assert cands == int(((d.flags & co.FLAG_VALID) != 0).sum()), (cands, d.flags)
        if prune:
            assert steps <= cands * nseg_pad, (steps, cands, nseg_pad)
            acc["pruned_steps"] = acc.get("pruned_steps", 0) + steps
            acc["full_steps"] = acc.get("full_steps", 0) + cands * nseg_pad
        else:
            assert steps == cands * nseg_pad, (steps, cands, nseg_pad)
        out.append(d)
    eng.configure(prune_window=0)
    return out


@gpu
@pytest.mark.parametrize("name", TRACKS)
def test_tracks_windows_poses(name):
    """every window on every track, poses whose i_ego puts the window across the seam on either
    side (on the raceline and 0.5 m off), random poses, and goals past the window's far end"""
    track = tracks()[name]
    eng = _engine(track)
    rng = np.random.default_rng(track.shape[0])
    acc = {}
    for W in windows(name):
        eng.configure(window=W)
        _, Wr = window_rule(track.shape[0], W, 0)
        poses = np.concatenate([ego_poses(track, Wr, rng), synth.scenario_batch(track, 3, 0, W + 7)[0]])
        for p in poses:
            _plan(eng, track, p, W, acc)
        if W in (1, 32, 129, 0):
            for p in poses[::3]:
                _plan(eng, track, p, W, acc, goals=GOALS)
    for cls in EGO_CLASSES:
        if not (name == "dup" and cls == "0"):   # nobody's nearest segment is a point
            assert acc["ego"].get(cls, 0) > 0, (name, cls, acc["ego"])
    assert acc["valid"] > 0
    _record("tracks_" + name, acc)


@gpu
@pytest.mark.parametrize("row", range(6))
def test_sample_count_shapes(row):
    """every sample count of shape_ms() on the ellipse (W = 128) and on the 2 cm track (W = 128:
    2.56 m, most samples beyond the far end); the G1-clothoid generator at the bucket's largest M;
    each launch confirmed through last_eval_shape"""
    r, ms = shape_ms()[row]
    acc = {"shapes": set()}
    for name in ("ellipse", "dense"):
        track = tracks()[name]
        eng = _engine(track)
        poses = np.concatenate([ego_poses(track, 128, np.random.default_rng(row))[::2],
                                synth.scenario_batch(track, 4, 0, 300 + row)[0]])
        for M in ms:
            for gen in ((0, 1) if M == r["m_max"] else (0,)):
                eng.configure(n_samples=M, generator=gen, window=128)
                for p in poses:
                    _plan(eng, track, p, 128, acc)
                    got = eng.last_eval_shape()
                    assert (got["ipl"], got["s"], got["sg"]) == (r["ipl"], r["s"], r["sg"]), (M, got, r)
                acc["shapes"].add("M=%d gen=%d split_odd=%d" % (M, gen, split_odd(r, M)))
        eng.close()
    _record("shapes_m%d" % r["m_max"], acc)


@gpu
def test_dense_lone_query_persistent_wide():
    """a lone query of 16 384 candidates at M = 200 on the 2 cm track: the persistent grid of the
    wide build; the deviation of 1024 candidates (and every other term of all) against the
    reference"""
    track = tracks()["dense"]
    eng = _engine(track, n_samples=200)
    eng.set_goal_grid(np.linspace(0.5, 6.0, 128), np.linspace(-1.2, 1.2, 128))
    pose = ego_poses(track, 128, np.random.default_rng(5))[2]
    d = eng.plan(pose, update_prev=False, want_states=True)
    got = eng.last_eval_shape()
    want = eval_choice(16384, 1, 200, 0, True)
    assert got["persistent"] == 1 and (got["nw"], got["minb"]) == (want["nw"], want["minb"]), (got, want)
    sel = np.sort(np.random.default_rng(1).choice(16384, 1024, replace=False))
    sub = d._replace(terms=d.terms[sel], flags=d.flags[sel], params=d.params[sel], states=d.states[sel])
    acc = {"instance": got["name"]}
    check_query(eng, track, pose, sub, 128, acc)
    _record("dense_persistent", acc)


@gpu
def test_colliding_candidates():
    """opponents and the corridor map: per-term costs are asked for, so colliding candidates keep
    their deviation, with the pruned scan too (which would skip them otherwise)"""
    track = tracks()["ellipse"]
    occ, origin, res = synth.corridor_grid()
    eng = _engine(track, kappa_max=3.0)
    eng.set_grid(occ, origin, res)
    eng.set_goal_grid(np.linspace(0.6, 4.0, 8), np.linspace(-2.0, 2.0, 9))
    acc = {"collide": 0}
    poses, opp, n_opp = synth.scenario_batch(track, 12, 8, 41)
    for p, o, k in zip(poses, opp, n_opp):
        for d in _plan(eng, track, p, 128, acc, opp=o[:k]):
            acc["collide"] += int((((d.flags & co.FLAG_VALID) != 0) & ((d.flags & 6) != 0)).sum())
    assert acc["collide"] > 0, acc
    _record("collisions", acc)


@gpu
@pytest.mark.parametrize("M", [33, 100])
def test_similarity(M):
    """rough previous paths (a one-sample shift shows) with every (n_shift, n_cull) kind: the
    default, none, a shift of one, one term, an empty range and a negative one; no previous path"""
    track = tracks()["ellipse"]
    eng = _engine(track, n_samples=M)
    rng = np.random.default_rng(M)
    prev = rng.uniform(-np.pi, np.pi, M).astype(np.float32)
    poses = synth.scenario_batch(track, 3, 0, M)[0]
    acc = {}
    for n_shift, n_cull in ((5, 10), (0, 0), (1, 0), (0, M - 1), (M // 2, M - M // 2), (M, 5)):
        eng.configure(n_shift=n_shift, n_cull=n_cull)
        eng.set_prev_path(prev)
        for p in poses:
            _plan(eng, track, p, 128, acc, prev=prev)
    eng.set_prev_path(None)
    for p in poses:
        _plan(eng, track, p, 128, acc)
    assert acc["valid"] > 0
    _record("similarity_m%d" % M, acc)


@gpu
def test_largest_window():
    """the largest window each reached single-query instance holds, on the 2 cm track"""
    import torch
    track = tracks()["dense"]
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    acc = {"shapes": set()}
    eng = _engine(track)
    for r, ms in shape_ms():
        M = r["m_max"]
        wmax = eval_choice(len(LA) * len(WD), 1, M, 0, True, False, sm)["max_window"]
        assert wmax < track.shape[0] - 1
        eng.configure(n_samples=M, window=wmax)
        for p in ego_poses(track, wmax, np.random.default_rng(M))[::4]:
            _plan(eng, track, p, wmax, acc)
        acc["shapes"].add("M=%d W=%d %s" % (M, wmax, eng.last_eval_shape()["name"]))
    _record("largest_window", acc)
