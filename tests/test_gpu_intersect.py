"""Every device intersect_point against the oracle's sequential scan (utils/utils.py:69-151).

The device runs intersect_point in five places: the free function (intersect_batch_kernel), the
pure-pursuit finish (sequential scan behind the FP32 TrackPrefilter), the sampler (8-lane group
scan of the first 32 segments, a 32-lane scan that resumes at segment 32, and a closing-segment-only
test for circles that stay clear of the raceline) and the planner's tracker (warp scan on the
float32 winning trajectory).  Every one evaluates a segment with the reference's float64 operations
in the oracle's order, so for the same input the hit (found, segment) must be identical and t and
the point bit-identical: only a shortcut can make them differ.  The queries here are aimed, with the
oracle, at the places where a shortcut can go wrong: hits 31 / 32 / 33 segments ahead, hits in the
wrap loop (closing segment and beyond), circles within millimetres of tangency or of the clear
threshold, open and sparse tracks and a large map origin.  test_crafted_queries_reach_every_class
(no GPU) keeps that coverage from being edited away.
"""
import functools
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from oracle import c_oracle as co
from tests import helpers as H

gpu = pytest.mark.gpu

OFFSETS = (0, 1, 7, 8, 9, 31, 32, 33, 63, 64)   # hit segment - int(t); plus a class ">=100"
DELTAS_MM = (-3.0, -1.0, -0.1, 0.1, 1.0, 1.9, 2.1, 3.0)   # nearest distance - L
PP_LOOKAHEADS = (0.3, 0.8, 2.0, 6.0, 15.0)
SAMPLER_LA = np.linspace(0.3, 9.0, 45)        # 45 rows: ragged over the sampler's 4 rows per warp
SAMPLER_WD = np.array([-0.6, 0.0, 0.6])


# -- tracks -----------------------------------------------------------------------------------
def _track(x, y, speed=6.0):
    """[n,5] (x, y, v, psi, kappa) with forward-difference headings; asserts no zero-length segment"""
    dx, dy = np.roll(x, -1) - x, np.roll(y, -1) - y
    assert (np.hypot(dx, dy)[:-1] > 1e-3).all()
    psi = np.mod(np.arctan2(dy, dx), 2.0 * np.pi)
    v = speed + 0.5 * np.sin(np.arange(x.size) * 0.37)   # distinct speeds: a wrong centre shows
    return np.stack([x, y, v, psi, np.zeros_like(x)], axis=1)


@functools.lru_cache(maxsize=None)
def tracks():
    rng = np.random.default_rng(2024)
    out = {"ellipse": synth.ellipse_track(),                        # closed, ~0.19 m segments
           "dense": synth.ellipse_track(n=20000)}                    # ~2 cm segments
    phi = np.sort(rng.uniform(0.0, 1.5 * np.pi, 257))               # open, irregular 1.5 pi arc:
    out["arc"] = _track(12.0 * np.cos(phi), 7.0 * np.sin(phi), 3.0)  # its closing segment is a chord
    phi = 2.0 * np.pi * (np.arange(100) + rng.uniform(-0.3, 0.3, 100)) / 100   # ~5 km, ~50 m segments
    out["sparse"] = _track(1000.0 * np.cos(phi) + 60.0 * np.cos(3 * phi),
                           600.0 * np.sin(phi) + 40.0 * np.sin(2 * phi), 20.0)
    for n in (3, 9, 33):                                             # one partial block
        phi = 2.0 * np.pi * np.arange(n) / n
        out["small%d" % n] = _track(8.0 * np.cos(phi), 5.0 * np.sin(phi))
    e = synth.ellipse_track().copy()
    e[:, 0] += 3000.0
    e[:, 1] -= 2000.0
    out["offset"] = e                                                # a map frame with a large origin
    return out


TRACKS = ("ellipse", "dense", "arc", "sparse", "small3", "small9", "small33", "offset")


def _normals(track):
    """left unit normal of every open segment and its length"""
    d = np.diff(track[:, :2], axis=0)
    ln = np.hypot(d[:, 0], d[:, 1])
    return np.stack([-d[:, 1], d[:, 0]], axis=1) / ln[:, None], ln


# -- oracle, threaded -------------------------------------------------------------------------
def _pmap(fn, n):
    with ThreadPoolExecutor(co.max_threads()) as ex:
        return list(ex.map(fn, range(n)))


def oracle_intersect(track, pts, t, radius, wrap):
    """co.intersect_point per query -> (found [m] bool, i [m], out [m,3] = px, py, t)"""
    radius = np.broadcast_to(np.asarray(radius, dtype=np.float64), (len(pts),))
    wrap = np.broadcast_to(np.asarray(wrap, dtype=bool), (len(pts),))
    found, idx, out = np.zeros(len(pts), bool), np.zeros(len(pts), np.int64), np.zeros((len(pts), 3))
    xy = np.ascontiguousarray(track[:, :2])

    def one(k):
        p, i, tt = co.intersect_point(pts[k], radius[k], xy, t[k], bool(wrap[k]))
        if p is not None:
            found[k], idx[k] = True, i
            out[k] = (p[0], p[1], tt)
    _pmap(one, len(pts))
    return found, idx, out


def hit_class(found, i, start_i):
    """offset class of one oracle answer"""
    if not found:
        return "miss"
    if i == -1:
        return "wrap:closing"
    if i < start_i:
        return "wrap:open"
    k = i - start_i
    if k in OFFSETS:
        return "k=%d" % k
    return "k>=100" if k >= 100 else "k:other"


def _classes(found, idx, t):
    out = {}
    for f, i, tt in zip(found, idx, t):
        c = hit_class(f, i, int(tt))
        out[c] = out.get(c, 0) + 1
    return out


# -- crafting ---------------------------------------------------------------------------------
def _crossings(track, P, R):
    """[m, n] bool: the circle (P[k], R[k]) has a root of the reference's quadratic in [0, 1] on
    segment i (column n-1: the closing segment), by the oracle's formulas in numpy.  Only aims the
    crafted queries; the oracle decides."""
    s = track[:, :2]
    e = np.roll(s, -1, axis=0) + 1e-6
    v = e - s
    a = (v * v).sum(1)
    d = s[None] - P[:, None]
    b = 2.0 * (v[None] * d).sum(2)
    c = (d * d).sum(2) - (R * R)[:, None]
    disc = b * b - 4.0 * a * c
    sq = np.sqrt(np.maximum(disc, 0.0))
    t1, t2 = (-b - sq) / (2.0 * a), (-b + sq) / (2.0 * a)
    return (disc >= 0) & (((t1 >= 0) & (t1 <= 1)) | ((t2 >= 0) & (t2 <= 1)))


def _radii(name, track):
    _, ln = _normals(track)
    r = [0.3, 0.8, 2.0, 6.0, 15.0]
    if ln.mean() > 10.0:
        r += [60.0, 400.0]
    return r


def _near(track, rng, m, spread, seam=False, lat=None):
    """m points scattered up to `spread` m off the raceline (near the seam if `seam`), or at the
    lateral offsets `lat`"""
    nrm, ln = _normals(track)
    nseg = ln.size
    j = rng.integers(max(0, nseg - 40), nseg, m) if seam else rng.integers(0, nseg, m)
    if seam:
        j[::2] = rng.integers(0, min(40, nseg), (m + 1) // 2)
    u = rng.uniform(0.0, 1.0, m)
    foot = track[j, :2] + u[:, None] * (track[j + 1, :2] - track[j, :2])
    lat = rng.uniform(-spread, spread, m) if lat is None else lat
    return foot + lat[:, None] * nrm[j]


@functools.lru_cache(maxsize=None)
def crafted_intersect(name):
    """intersect_point queries aimed at every offset class and both wrap cases:
    {(radius, wrap): (points [m,2], t [m])}"""
    track = tracks()[name]
    n = track.shape[0]
    rng = np.random.default_rng(len(name) * 7919 + n)
    sets = {}
    for R in _radii(name, track):
        P = np.concatenate([_near(track, rng, 60, 1.5 * R), _near(track, rng, 40, 1.5 * R, seam=True),
                            _tangent_points(track, rng, R, 4), _aimed_at_seam(track, rng, R, 40)])
        cr = _crossings(track, P, np.full(len(P), R))
        op = cr[:, :n - 1]
        pts, ts, wr = [], [], []
        for p in range(len(P)):
            hs = np.nonzero(op[p])[0]
            prev = -1
            for h in hs[:6]:
                gap = h - prev - 1          # free segments before the crossing h
                prev = h
                ks = [k for k in OFFSETS if k <= gap]
                if gap >= 100:
                    ks.append(int(rng.integers(100, gap + 1)))
                for k in ks:
                    u = 0.0 if (k == 0 or rng.random() < 0.4) else rng.uniform(0.0, 1.0)
                    pts.append(P[p]); ts.append(h - k + u); wr.append(bool(rng.integers(0, 2)))
            # forward scan empty from `start` on: the wrap loop decides (closing segment or beyond)
            last = hs[-1] if hs.size else -1
            lo = max(last + 1, n - 41)
            if lo <= n - 2:
                for start in {lo, n - 2, int(rng.integers(lo, n - 1))}:
                    u = 0.0 if rng.random() < 0.3 else rng.uniform(0.0, 1.0)
                    pts.append(P[p]); ts.append(start + u); wr.append(True)
                    pts.append(P[p]); ts.append(start + u); wr.append(False)
        pts, ts, wr = np.array(pts).reshape(-1, 2), np.array(ts), np.array(wr, bool)
        for w in (False, True):
            sets[(R, w)] = (np.ascontiguousarray(pts[wr == w]), ts[wr == w])
    return sets


def _aimed_at_seam(track, rng, R, m):
    """m points at distance R behind (along the raceline) a point of the closing segment or of a
    segment within 3 of the seam: circles that cross the track there"""
    n = track.shape[0]
    j = rng.integers(-3, 4, m) % n                        # segment j: waypoint j -> j + 1 (mod n)
    s, e = track[j, :2], track[(j + 1) % n, :2]
    x = s + rng.uniform(0.0, 1.0, m)[:, None] * (e - s)
    u = (e - s) / np.hypot(*(e - s).T)[:, None]
    a = rng.normal(0.0, 0.2, m)
    back = np.stack([u[:, 0] * np.cos(a) - u[:, 1] * np.sin(a), u[:, 0] * np.sin(a) + u[:, 1] * np.cos(a)], 1)
    return x - R * back


def _tangent_points(track, rng, L, per_delta, seam=False):
    """points whose distance to segment j (at an interior foot) is L + delta, on both sides"""
    nrm, ln = _normals(track)
    nseg = ln.size
    out = []
    for d in DELTAS_MM:
        j = rng.integers(0, nseg, per_delta)
        if seam:
            j = np.where(rng.random(per_delta) < 0.5, rng.integers(max(0, nseg - 5), nseg, per_delta),
                         rng.integers(0, min(5, nseg), per_delta))
        u = rng.uniform(0.2, 0.8, per_delta)
        side = np.where(np.arange(per_delta) % 2 == 0, 1.0, -1.0)
        foot = track[j, :2] + u[:, None] * (track[j + 1, :2] - track[j, :2])
        out.append(foot + (side * (L + 1e-3 * d))[:, None] * nrm[j])
    return np.concatenate(out)


def random_intersect(name, m, seed):
    """m random (point, t, radius) queries per radius and wrap: t = 0, integers, the last segment
    [n-2, n-1) or anywhere"""
    track = tracks()[name]
    n = track.shape[0]
    rng = np.random.default_rng(seed)
    lo, hi = track[:, :2].min(0), track[:, :2].max(0)
    sets = {}
    for R in _radii(name, track):
        for w in (False, True):
            P = np.concatenate([_near(track, rng, m // 2, 1.5 * R),
                                rng.uniform(lo - R, hi + R, (m - m // 2, 2))])
            t = rng.uniform(0.0, n - 1.0, m)
            kind = rng.integers(0, 4, m)
            t[kind == 0] = 0.0
            t[kind == 1] = np.floor(t[kind == 1])
            t[kind == 2] = n - 2 + rng.uniform(0.0, 1.0, (kind == 2).sum())
            sets[(R, w)] = (P, t)
    return sets


@functools.lru_cache(maxsize=None)
def crafted_poses(name, L):
    """pure-pursuit poses [m,3]: nearest distance L + delta (both sides, also at the seam), random
    lateral offsets up to 1.5 L, and poses at the seam"""
    track = tracks()[name]
    rng = np.random.default_rng(int(L * 1000) + track.shape[0])
    xy = np.concatenate([_tangent_points(track, rng, L, 10), _tangent_points(track, rng, L, 2, seam=True),
                         _near(track, rng, 300, max(1.5 * L, 1.0)),
                         _near(track, rng, 60, max(1.5 * L, 1.0), seam=True)])
    return np.concatenate([xy, rng.uniform(-np.pi, np.pi, (len(xy), 1))], axis=1)


def _nearest_dist(track, xy):
    d = np.zeros(len(xy))
    base = np.ascontiguousarray(track[:, :2])

    def one(k):
        d[k] = co.nearest_point(xy[k], base)[1]
    _pmap(one, len(xy))
    return d


@functools.lru_cache(maxsize=None)
def sampler_poses(name):
    """planner poses [m,4]: random, at the clear threshold of chosen rows (nearest distance
    L_row + delta), at the seam and, on the open arc, around the closing chord"""
    track = tracks()[name]
    rng = np.random.default_rng(track.shape[0] + 77)
    # lateral offsets 0..0.6 m move the hit of each row continuously: on the 2 cm track the rows
    # near L = 0.7 m then land 31, 32 and 33 segments ahead
    xy = [_near(track, rng, 10, 1.0), _near(track, rng, 4, 1.0, seam=True),
          _near(track, rng, 12, 0.0, lat=np.linspace(0.0, 0.6, 12))]
    for row in (0, 13, 30):
        xy.append(_tangent_points(track, rng, SAMPLER_LA[row], 1))
    if name == "arc":
        a, b = track[-1, :2], track[0, :2]
        f = rng.uniform(0.3, 0.7, 6)
        xy.append(a + f[:, None] * (b - a) + rng.normal(0.0, 0.3, (6, 2)))
    xy = np.concatenate(xy)
    th = rng.uniform(-np.pi, np.pi, len(xy))
    return np.concatenate([xy, th[:, None], rng.uniform(2.0, 8.0, (len(xy), 1))], axis=1)


def sampler_classes(name):
    """oracle answer of every (pose, row) of sampler_poses: {class: count}, with 'clear:closing'
    for a row whose circle stays clear of the raceline (d > L + 2 mm) and hits the closing segment"""
    track = tracks()[name]
    poses = sampler_poses(name)
    base = np.ascontiguousarray(track[:, :2])
    counts = {}
    for p in poses:
        _, d, t, i = co.nearest_point(p[:2], base)
        for L in SAMPLER_LA:
            q, hi, _ = co.intersect_point(p[:2], L, base, i + t, True)
            c = hit_class(q is not None, hi, i)
            counts[c] = counts.get(c, 0) + 1
            if d > L + 2e-3 and q is not None and hi == -1:
                counts["clear:closing"] = counts.get("clear:closing", 0) + 1
            if abs(d - L) < 2e-3:
                key = "tangent:<L" if d < L else "tangent:>=L"
                counts[key] = counts.get(key, 0) + 1
    return counts


# -- coverage (no GPU) ------------------------------------------------------------------------
def test_crafted_queries_reach_every_class():
    """The crafted sets reach, by the oracle's answer, every hit offset (including 31 / 32 / 33
    around the sampler's group-scan boundary and >= 100) on the two ellipses, both wrap cases on
    every closed track with enough segments, tangent circles within 2 mm on both sides, a clear
    sampler row that hits the open arc's closing segment, and sampler hits 31..33 segments ahead."""
    record = {}
    for name in ("ellipse", "dense", "offset", "sparse"):
        cls = {}
        for (R, w), (P, t) in crafted_intersect(name).items():
            f, i, _ = oracle_intersect(tracks()[name], P, t, R, w)
            for c, v in _classes(f, i, t).items():
                cls[c] = cls.get(c, 0) + v
        record["A:" + name] = cls
        need = ["wrap:closing", "wrap:open", "k=0", "k=1"]
        if name in ("ellipse", "dense", "offset"):
            need += ["k=%d" % k for k in OFFSETS] + ["k>=100"]
        for c in need:
            assert cls.get(c, 0) > 0, (name, c, cls)
    for name in ("ellipse", "arc", "sparse"):
        for L in (0.3, 6.0):
            P = crafted_poses(name, L)
            d = _nearest_dist(tracks()[name], P[:, :2])
            tb = int(((d - L > -2e-3) & (d < L)).sum()), int(((d >= L) & (d - L < 2e-3)).sum())
            record["B:%s:L=%g:tangent(<L,>=L)" % (name, L)] = list(tb)
            assert tb[0] > 0 and tb[1] > 0, (name, L, tb)
    for name in ("ellipse", "dense", "arc"):
        cls = sampler_classes(name)
        record["C:" + name] = cls
        assert cls.get("tangent:<L", 0) > 0 and cls.get("tangent:>=L", 0) > 0, (name, cls)
        if name == "arc":
            assert cls.get("clear:closing", 0) > 0, cls
        else:
            for c in ("k=31", "k=32", "k=33"):
                assert cls.get(c, 0) > 0, (name, c, cls)
    H.record_parity("intersect_crafted_classes", record)


# -- A. intersect_point_batch -----------------------------------------------------------------
def _engine(track, **cfg):
    from f1tenth_planning_b200.engine import Engine
    eng = Engine(**cfg)
    eng.set_track(track)
    return eng


def _check_intersect(eng, track, P, t, R, w):
    out, oi = eng.intersect_point_batch(P, t, R, w)
    f, i, o = oracle_intersect(track, P, t, R, w)
    assert np.array_equal(out[:, 3] != 0, f), ("found", R, w, np.nonzero((out[:, 3] != 0) != f)[0][:5])
    assert np.array_equal(oi[f], i[f]), ("segment", R, w)
    assert np.array_equal(out[f, :3], o[f][:, [0, 1, 2]]), ("t / point", R, w)
    return f, i


@gpu
def test_intersect_batch_golden(golden_spielberg, golden_misc):
    """the 300 golden rows minted from the reference, one call per distinct (radius, wrap)"""
    m, wp = golden_misc, golden_spielberg["waypoints"]
    eng = _engine(wp)
    done = 0
    for R in np.unique(m["ip_radius"]):
        for w in (False, True):
            sel = np.nonzero((m["ip_radius"] == R) & (m["ip_wrap"] == w))[0]
            if sel.size == 0:
                continue
            out, oi = eng.intersect_point_batch(m["ip_points"][sel], m["ip_t"][sel], R, w)
            found = m["ip_out"][sel, 3] != 0
            assert np.array_equal(out[:, 3] != 0, found)
            assert np.array_equal(oi[found], m["ip_i"][sel][found])
            # the reference's numpy arithmetic, not pinned to the operation order: 1e-9 (its value
            # against the oracle, which is, is bit for bit below)
            np.testing.assert_allclose(out[found, :3], m["ip_out"][sel][found, :3], rtol=0, atol=1e-9)
            _check_intersect(eng, wp, m["ip_points"][sel], m["ip_t"][sel], R, w)
            done += sel.size
    assert done == 300


@gpu
@pytest.mark.parametrize("name", TRACKS)
def test_intersect_batch_crafted_and_random(name):
    track = tracks()[name]
    eng = _engine(track)
    cls, total = {}, 0
    sets = list(crafted_intersect(name).items()) + list(random_intersect(name, 1000, 11).items())
    for (R, w), (P, t) in sets:
        f, i = _check_intersect(eng, track, P, t, R, w)
        for c, v in _classes(f, i, t).items():
            cls[c] = cls.get(c, 0) + v
        total += len(P)
    assert total >= 10000
    cls["queries"] = total
    cls["mismatch"] = 0
    H.record_parity("intersect_A_" + name, cls)


# -- B. pure pursuit --------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", TRACKS)
def test_pure_pursuit_lookaheads(name):
    """every lookahead column, lookahead_i and status against the oracle; vertex ties (the FP32
    scan picks the neighbouring segment at the same distance) counted and excluded as in
    test_gpu_pure_pursuit._check; the device-tensor call is bit-identical to the host call"""
    import torch
    track = tracks()[name]
    eng = _engine(track)
    stats = {}
    for L in PP_LOOKAHEADS:
        poses = crafted_poses(name, L)
        r = eng.pure_pursuit_batch(poses, L)
        o = co.pure_pursuit_batch(track, poses, L, n_threads=co.max_threads())
        same = r.nearest_i == o["nearest_i"]
        st = stats.setdefault("L=%g" % L, {"poses": len(poses), "vertex_tie": 0, "flat_minimum": 0})
        for k in np.nonzero(~same)[0]:
            gi, oi = int(r.nearest_i[k]), int(o["nearest_i"][k])
            gd, od = r.nearest[k, 2], o["nearest"][k, 2]
            if abs(gi - oi) == 1 and abs(gd - od) < 1e-9:
                st["vertex_tie"] += 1          # (k, t=1) == (k+1, t=0)
            else:
                # a pose near a centre of curvature of a 2 cm raceline: the distance is flat over
                # several segments, below the FP32 scan's resolution (nearest_point's own tests)
                assert od <= gd <= od + 1e-6 * max(od, 1.0), (L, k, gi, oi, gd, od)
                st["flat_minimum"] += 1
        assert (~same).mean() < 0.02, (L, (~same).mean())
        np.testing.assert_allclose(r.nearest[same], o["nearest"][same], rtol=1e-9, atol=1e-9)
        assert np.array_equal(r.status, o["status"]), (L, np.nonzero(r.status != o["status"])[0][:5])
        assert np.array_equal(r.lookahead[same], o["lookahead"][same]), L
        assert np.array_equal(r.lookahead_i[same], o["lookahead_i"][same]), L
        np.testing.assert_allclose(r.actuation[same], o["actuation"][same], rtol=0, atol=1e-12)
        d = o["nearest"][:, 2]
        st["found"] = int((o["lookahead"][:, 3] > 0).sum())
        st["tangent<2mm"] = int((np.abs(d - L) < 2e-3).sum())
        st["status"] = [int((o["status"] == s).sum()) for s in (0, 1, 2)]
        # the device-tensor entry point on the same poses
        dev = torch.device("cuda", eng.device)
        B = len(poses)
        t = dict(nearest=torch.zeros(B, 4, dtype=torch.float64, device=dev),
                 nearest_i=torch.zeros(B, dtype=torch.int32, device=dev),
                 lookahead=torch.zeros(B, 4, dtype=torch.float64, device=dev),
                 lookahead_i=torch.zeros(B, dtype=torch.int32, device=dev),
                 actuation=torch.zeros(B, 2, dtype=torch.float64, device=dev),
                 status=torch.zeros(B, dtype=torch.int32, device=dev))
        eng.pure_pursuit_batch_dev(torch.from_numpy(poses).to(dev), L, **t)
        torch.cuda.synchronize(dev)
        for k, v in t.items():
            assert np.array_equal(v.cpu().numpy(), getattr(r, k)), (L, k)
    H.record_parity("intersect_B_" + name, stats)


# -- C. sampler -------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", TRACKS)
def test_sampler_centres(name):
    """NO_CENTRE flags of every lookahead row exactly the oracle's and the goals within 1e-5 (a
    wrong centre moves a goal by a segment, >= 2 cm here); the batch path bit-identical to the
    single queries; one row-sharded call gives the same flags on its rows"""
    track = tracks()[name]
    eng, cfg, world = H.make_pair(track, SAMPLER_LA, SAMPLER_WD, kappa_max=0.0)
    eng.set_prev_path(None)
    poses = sampler_poses(name)
    nc = {"poses": len(poses), "no_centre": 0, "rows": len(poses) * len(SAMPLER_LA)}
    single = []
    for p in poses:
        d = eng.plan(p, update_prev=False)
        o = co.plan(cfg, world, p)
        gf, of = d.flags & co.FLAG_NO_CENTRE, o["flags"] & co.FLAG_NO_CENTRE
        assert np.array_equal(gf, of), (name, p, np.nonzero(gf != of)[0][:6])
        ok = of == 0
        assert H.close(d.goals[ok], o["goals"][ok], 1e-5, 1e-5).all(), (name, p)
        nc["no_centre"] += int((~ok).sum()) // len(SAMPLER_WD)
        single.append(d)
    b = eng.plan_batch(poses, want_flags=True)
    ob = co.plan_batch(cfg, world, poses, n_threads=co.max_threads())
    assert np.array_equal(b.flags & co.FLAG_NO_CENTRE, ob["flags"] & co.FLAG_NO_CENTRE)
    for s, d in enumerate(single):
        assert np.array_equal(b.costs[s], d.costs), (name, s)
        assert np.array_equal(b.flags[s], d.flags), (name, s)
    W = 4
    r = 1
    d = eng.plan(poses[-1], update_prev=False, rows=(r, W))
    mine = np.zeros((len(SAMPLER_LA), len(SAMPLER_WD)), bool)
    mine[r::W] = True
    assert np.array_equal(d.flags[mine.ravel()], single[-1].flags[mine.ravel()])
    nc.update(sampler_classes(name))
    H.record_parity("intersect_C_" + name, nc)


# -- D. tracker -------------------------------------------------------------------------------
def _tracker_reference(traj, pose, v_goal, literal, L, wb, max_reacquire):
    """pure pursuit on the device's own float32 winning trajectory, widened exactly: the rules of
    select_kernel's tracker (lattice_planner.py:208-212) with the oracle's float64 functions"""
    xy = np.ascontiguousarray(traj[:, :2].astype(np.float64))
    M = xy.shape[0]
    q = np.array(pose[:2], dtype=np.float64) if literal else np.zeros(2)
    qth = float(pose[2]) if literal else 0.0
    wb = 0.33 if literal else wb            # the literal tracker is built with the default
    _, d, t, i = co.nearest_point(q, xy)
    speed = float(traj[i, 2]) if literal else v_goal
    if d < L:
        p, hi, _ = co.intersect_point(q, L, xy, i + t, True)
        if p is None:
            return 0, 0.0, 0.0
        lp = xy[hi % M]
    elif d < max_reacquire:
        lp = xy[i]
    else:
        return 0, 0.0, 0.0
    _, steer = co.get_actuation(qth, [lp[0], lp[1], speed], q, L, wb)
    return 1, steer, speed


@gpu
@pytest.mark.parametrize("literal", [0, 1])
def test_tracker_teacher_forced(literal):
    """the planner's tracker on its own best_traj: tracker_found exact, steer within 1e-12, speed
    exact; batch steer_speed bit-identical to the single query.  The ellipse is shifted so that it
    passes the map origin: the literal tracker queries the map-frame pose against the vehicle-frame
    trajectory, and only there does its circle reach the trajectory."""
    track = synth.ellipse_track().copy()
    track[:, 0] -= 80.0
    track[:, 2] += 0.25 * np.sin(np.arange(track.shape[0]) * 0.1)   # a wrong centre shows in speed
    la, wd = np.array([0.6, 1.2, 1.8, 2.4]), np.linspace(-0.8, 0.8, 5)
    eng, cfg, world = H.make_pair(track, la, wd, kappa_max=0.0, literal_tracker=literal)
    eng.set_prev_path(None)
    rng = np.random.default_rng(91 + literal)
    n = track.shape[0]
    j = np.concatenate([rng.integers(n - 25, n, 8), rng.integers(0, 25, 8), rng.integers(0, n, 8)])
    lat = rng.uniform(-0.6, 0.6, j.size)
    psi = track[j, 3]
    poses = np.stack([track[j, 0] - lat * np.sin(psi), track[j, 1] + lat * np.cos(psi),
                      psi + rng.normal(0.0, 0.15, j.size), rng.uniform(2.0, 8.0, j.size)], axis=1)
    base = np.ascontiguousarray(track[:, :2])
    stats = {}
    for L in (0.3, 0.8, 2.5, 50.0):   # 50 m: longer than any winning trajectory
        eng.configure(tracker_lookahead=L)
        st = stats.setdefault("L=%g" % L, {"found": 0, "not_found": 0})
        single = []
        for p in poses:
            d = eng.plan(p, update_prev=False)
            # v_goal: the raceline speed at the winner's goal centre (lattice_planner.py:249-251)
            _, _, t0, i0 = co.nearest_point(p[:2], base)
            hp, hi, _ = co.intersect_point(p[:2], la[d.best_idx // len(wd)], base, i0 + t0, True)
            v_goal = float(track[hi % n, 2]) if hp is not None else float(p[3])
            f, steer, speed = _tracker_reference(d.best_traj, p, v_goal, literal, L,
                                                 eng.config.wheelbase, eng.config.max_reacquire)
            assert int(d.tracker_found) == f, (L, p)
            assert abs(d.steer - steer) <= 1e-12, (L, p, d.steer, steer)
            assert d.speed == speed, (L, p, d.speed, speed)
            st["found" if f else "not_found"] += 1
            single.append((d.steer, d.speed))
        b = eng.plan_batch(poses)
        assert np.array_equal(b.steer_speed, np.array(single)), L
    H.record_parity("intersect_D_literal%d" % literal, stats)


# -- E. get_actuation_batch -------------------------------------------------------------------
@gpu
def test_actuation_batch_golden_and_threshold(golden_misc):
    """the 64 golden rows in one call, and rows whose lateral offset wy straddles the 1e-6
    threshold below which the reference steers straight"""
    rng = np.random.default_rng(5)
    m = 400
    th = rng.uniform(-np.pi, np.pi, m)
    pos = rng.uniform(-5.0, 5.0, (m, 2))
    fwd = rng.uniform(0.2, 3.0, m)
    # |wy| - 1e-6 between 1e-14 and 1e-12, either side: wider than the ~1e-16 m the two sides'
    # sin / cos may move wy by, so the decision is the same on both
    eps = 10.0 ** rng.uniform(-8, -6, m) * np.where(rng.random(m) < 0.5, 1.0, -1.0)
    wy = 1e-6 * (1.0 + eps) * np.where(np.arange(m) % 2 == 0, 1.0, -1.0)
    c, s = np.cos(th), np.sin(th)
    lp = pos + np.stack([c * fwd - s * wy, s * fwd + c * wy], axis=1)
    rows = np.concatenate([golden_misc["act_in"],
                           np.stack([th, lp[:, 0], lp[:, 1], rng.uniform(1, 8, m), pos[:, 0], pos[:, 1],
                                     rng.uniform(0.3, 3.0, m)], axis=1)])
    eng = _engine(tracks()["ellipse"])
    out = eng.get_actuation_batch(rows, 0.33)
    ref = np.array([co.get_actuation(r[0], r[1:4], r[4:6], r[6], 0.33) for r in rows])
    assert np.array_equal(out[:, 0], ref[:, 0])
    np.testing.assert_allclose(out[:, 1], ref[:, 1], rtol=0, atol=1e-12)
    np.testing.assert_allclose(out[:64], golden_misc["act_out"], rtol=1e-12, atol=1e-12)
    straight = ref[64:, 1] == 0.0
    H.record_parity("intersect_E_actuation", {"rows": int(rows.shape[0]),
                                             "threshold_straight": int(straight.sum()),
                                             "threshold_steered": int((~straight).sum())})
    assert straight.any() and (~straight).any()
