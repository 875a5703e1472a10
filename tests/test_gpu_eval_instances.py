"""Every eval_kernel instance the launch policy can pick, at the sample counts where its tiling
changes (the bucket edges of the instance table and the odd-row edges of the S = 13 shapes).

For each M: single queries against the float64 oracle (and the float32 collision mirror, and the
generator against the oracle's spiral); then every regime the library's own choice function
(f1l_debug_eval_choice) lists as reachable for the bucket -- each workload confirmed through
last_eval_shape -- bit for bit against single queries on the same scenarios, with the PW twin of
every batch regime; dense lone queries against their row and block shards.  Once per bucket:
pruned against full window scans, the G1-clothoid generator, disc collisions, the dense regimes
against oracle slices, and the largest window of every reachable instance."""
import numpy as np
import pytest

from f1tenth_planning_b200 import synth
from f1tenth_planning_b200._lib import F1LError
from oracle import c_oracle as co
from tests import helpers as H
from tests.test_eval_choice import eval_builds, eval_choice, instance, reachable
from tests.test_gpu_batch_weights import _weight_rows

pytestmark = pytest.mark.gpu

MS = [2, 3, 31, 32, 33, 63, 64, 65, 96, 97, 100, 101, 104, 105, 127, 128, 129, 192, 193, 200, 201,
      208, 209, 255, 256]
ONCE = (32, 64, 104, 128, 208, 256)     # one M per bucket: its largest
RAGGED = (13, 25, 30, 256)              # candidate counts with a ragged last item of four
SAMPLER = (4, 5, 31, 32)                # scenario counts where the sampler changes its launch
N_SINGLE = 64                           # scenarios of a batch checked against single queries
K_OPP = 8
FIELDS = ("costs", "flags", "terms", "best_idx", "best_cost", "best_traj", "steer_speed")


def _sm(eng):
    import torch
    return torch.cuda.get_device_properties(eng.device).multi_processor_count


def _row(M):
    return next(r for r in eval_builds() if M <= r["m_max"])


def _grid(n):
    """a goal grid of exactly n candidates: nL lookahead rows x nW widths, nL <= nW"""
    nl = max(d for d in range(1, int(np.sqrt(n)) + 1) if n % d == 0)
    la = np.linspace(0.6, 3.6, nl) if nl > 1 else np.array([1.6])
    return la, np.linspace(-1.2, 1.2, n // nl) if n > nl else np.array([0.0])


def _engine(track, corridor, M, n, **cfg):
    la, wd = _grid(n)
    return H.make_pair(track, la, wd, grid=corridor, n_samples=M, **cfg)


def _world(eng, track, corridor, n):
    """an oracle world of the engine's goal grid of n candidates, seeded from the device LUT"""
    la, wd = _grid(n)
    lut, ranges = eng.get_lut()
    occ, origin, res = corridor
    return co.World_(track, la, wd, grid=occ, grid_origin=origin, grid_res=res, lut=lut, lut_ranges=ranges)


def _workloads(M, sm):
    """{instance: [(n_cand, S, lone), ...]} of every regime (persistent grid, candidates per pull)
    the choice function reaches at M with the cubic generator and without weights"""
    out = {}
    for key, (n, S, gen, lone, w) in sorted(reachable(M, sm).items()):
        if gen == 0 and not w:
            out.setdefault(key[:5], []).append((n, S, lone))
    return out


def _confirm(eng, n, S, M, sm, lone=False, weights=False):
    """the launch just made is the one the choice function names"""
    want = eval_choice(n, S, M, 0 if eng.config.generator == 0 else 1, lone, weights, sm)
    got = eng.last_eval_shape()
    row = _row(M)
    assert (got["ipl"], got["s"], got["sg"]) == (row["ipl"], row["s"], row["sg"]), (got, row)
    for k in ("nw", "minb", "chunk", "ctas_per_scenario", "item", "persistent", "pw"):
        assert got[k] == want[k], (k, n, S, M, lone, weights, got, want)
    return got


class _Batch:
    pass


def _batch_dev(eng, poses, opp, n_opp, weights=None, want_terms=True):
    """one batch call on device buffers (one launch of the pipeline over all S scenarios, unlike
    the host-buffer call, which runs chunks) -> numpy outputs"""
    import torch
    dev = torch.device("cuda", eng.device)
    S, C, M = poses.shape[0], eng.n_candidates, eng.n_samples
    o = dict(best_idx=torch.empty(S, dtype=torch.int32, device=dev),
             best_cost=torch.empty(S, dtype=torch.float32, device=dev),
             best_traj=torch.empty(S, M, 4, dtype=torch.float32, device=dev),
             costs=torch.empty(S, C, dtype=torch.float32, device=dev),
             flags=torch.empty(S, C, dtype=torch.uint8, device=dev),
             steer_speed=torch.empty(S, 2, dtype=torch.float64, device=dev),
             terms=torch.empty(S, C, 5, dtype=torch.float32, device=dev) if want_terms else None)
    w = None if weights is None else torch.from_numpy(np.ascontiguousarray(weights, np.float32)).to(dev)
    eng.plan_batch_dev(*(torch.from_numpy(a).to(dev) for a in (poses, opp, n_opp)), weights=w, **o)
    torch.cuda.synchronize(dev)
    b = _Batch()
    for k, v in o.items():
        setattr(b, k, None if v is None else v.cpu().numpy())
    return b


def _single_mismatches(eng, b, poses, opp, n_opp, idx, W=None):
    """scenarios of idx whose single query (after configure(weights=W[s]) when W is given) is not
    bit-identical to the batch row in any of FIELDS"""
    bad = []
    default = list(eng.config.weights)
    for s in idx:
        if W is not None:
            eng.configure(weights=W[s].astype(np.float64))
        d = eng.plan(poses[s], opp[s, :n_opp[s]], update_prev=False)
        same = (np.array_equal(d.costs, b.costs[s]) and np.array_equal(d.flags, b.flags[s])
                and np.array_equal(d.terms, b.terms[s]) and d.best_idx == b.best_idx[s]
                and np.float32(d.best_cost) == b.best_cost[s] and np.array_equal(d.best_traj, b.best_traj[s])
                and d.steer == b.steer_speed[s, 0] and d.speed == b.steer_speed[s, 1])
        if not same:
            bad.append(int(s))
    if W is not None:
        eng.configure(weights=default)
    return bad


def _batch_regime(eng, track, M, sm, n, S, seed, stats, name):
    """a batch regime and its PW twin against single queries; returns the instances it ran"""
    la, wd = _grid(n)
    eng.set_goal_grid(la, wd)
    eng.set_prev_path(None)
    poses, opp, n_opp = synth.scenario_batch(track, S, K_OPP, seed)
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(S, min(S, N_SINGLE), replace=False))
    b = _batch_dev(eng, poses, opp, n_opp)
    ran = [_confirm(eng, n, S, M, sm)["name"]]
    bad = _single_mismatches(eng, b, poses, opp, n_opp, idx)
    # PW twin: the config's weights broadcast change no bit; varied rows plan as the single query
    # configured with the row
    default = np.array(list(eng.config.weights), np.float32)
    bw = _batch_dev(eng, poses, opp, n_opp, weights=np.tile(default, (S, 1)))
    ran.append(_confirm(eng, n, S, M, sm, weights=True)["name"])
    broadcast = [k for k in FIELDS if not np.array_equal(getattr(bw, k), getattr(b, k))]
    W = _weight_rows(default, max(S, 22), seed)[:S]
    bv = _batch_dev(eng, poses, opp, n_opp, weights=W)
    bad_w = _single_mismatches(eng, bv, poses, opp, n_opp, idx, W)
    stats[name] = {"n_cand": n, "S": S, "instance": ran[0], "singles": len(idx), "mismatch": len(bad),
                   "pw_broadcast_fields_differ": broadcast, "pw_rows_mismatch": len(bad_w),
                   "finite": int(np.isfinite(b.costs[idx]).sum())}
    assert not bad and not broadcast and not bad_w, (name, stats[name], bad[:8], bad_w[:8])
    return ran


def _pieces(n, M, sm):
    """the fewest power-of-two shards whose queries run static (not persistent) grids"""
    k = 2
    while eval_choice(-(-n // k), 1, M, 0, True, False, sm)["persistent"]:
        k *= 2
    return k


def _dense_regime(eng, track, M, sm, n, seed, stats, name):
    """a lone dense query against its row and block shards, which run static grids"""
    la, wd = _grid(n)
    eng.set_goal_grid(la, wd)
    eng.set_prev_path(None)
    pose, opp = H.scenario(track, seed, K_OPP)
    whole = eng.plan(pose, opp, update_prev=False)
    got = _confirm(eng, n, 1, M, sm, lone=True)
    assert got["persistent"] == 1
    nl, nw = len(la), len(wd)
    k = _pieces(n, M, sm)
    bad = []
    for mode in ("rows", "blocks"):
        best, seen = [], np.zeros(n, bool)
        for r in range(min(k, nl) if mode == "rows" else k):
            if mode == "rows":
                step = min(k, nl)
                p = eng.plan(pose, opp, update_prev=False, rows=(r, step))
                mine = np.zeros((nl, nw), bool)
                mine[r::step] = True
                mine = mine.ravel()
            else:
                lo, hi = r * n // k, (r + 1) * n // k
                p = eng.plan(pose, opp, update_prev=False, shard=(lo, hi))
                mine = np.zeros(n, bool)
                mine[lo:hi] = True
            assert eng.last_eval_shape()["persistent"] == 0, (mode, r, eng.last_eval_shape())
            if not (np.array_equal(p.costs[mine], whole.costs[mine]) and np.array_equal(p.flags[mine], whole.flags[mine])
                    and np.array_equal(p.terms[mine], whole.terms[mine])):
                bad.append((mode, r))
            if mine[whole.best_idx] and np.isfinite(whole.best_cost):
                if not (p.best_idx == whole.best_idx and np.array_equal(p.best_traj, whole.best_traj)
                        and p.steer == whole.steer and p.speed == whole.speed):
                    bad.append((mode, r, "winner"))
            best.append((float(p.best_cost), int(p.best_idx)))
            seen |= mine
        assert seen.all()
        if np.isfinite(whole.best_cost) and min(best)[1] != whole.best_idx:
            bad.append((mode, "argmin"))
    stats[name] = {"n_cand": n, "instance": got["name"], "pieces": k, "mismatch": len(bad),
                   "finite": int(np.isfinite(whole.costs).sum())}
    assert not bad, (name, stats[name], bad[:8])
    return pose, opp, whole


def _oracle_slice(cfg, world, pose, opp, costs, flags, lo, hi, counts):
    """device costs / flags of candidates [lo, hi) against the oracle on that slice: every flag
    mismatch at a decision margin, finite costs within the parity tolerance"""
    o = co.plan(cfg, world, pose, opp, c_begin=lo, c_end=hi, want_states=True)
    C = costs.shape[0]
    osl = {k: (v[lo:hi] if isinstance(v, np.ndarray) and v.shape[:1] == (C,) else v) for k, v in o.items()}
    H.classify_flags(flags[lo:hi], osl, cfg, counts=counts)
    same = (flags[lo:hi] & 0xF) == (osl["flags"] & 0xF)
    assert (np.isfinite(osl["costs"]) == np.isfinite(costs[lo:hi]))[same].all()
    fin = np.isfinite(osl["costs"]) & np.isfinite(costs[lo:hi])
    assert H.close(costs[lo:hi][fin], osl["costs"][fin]).all()
    counts["candidates"] = counts.get("candidates", 0) + hi - lo
    counts["finite"] = counts.get("finite", 0) + int(fin.sum())


@pytest.mark.parametrize("M", MS)
def test_reference(ellipse, corridor, M):
    """single queries against the float64 oracle, the float32 collision mirror and the spiral"""
    eng, cfg, world = _engine(ellipse, corridor, M, 28, kappa_max=3.0)
    hl, hw = np.float32(0.5 * cfg.car_length), np.float32(0.5 * cfg.car_width)
    rc2 = np.float32(4.0 * ((0.5 * cfg.car_length) ** 2 + (0.5 * cfg.car_width) ** 2))
    stats = {"valid": 0, "mirror_mismatch": 0, "collide": 0}
    for seed in (3100 + M, 3400 + M, 3700 + M):
        pose, opp = H.scenario(ellipse, seed, K_OPP)
        d = eng.plan(pose, opp, update_prev=False, want_states=True, want_headings=True, want_map=True)
        o = co.plan(cfg, world, pose, opp, want_states=True)
        st = H.compare_plan(d, o, cfg)
        stats["both_valid"] = stats.get("both_valid", 0) + st["n_both_valid"]
        f, i = eng.debug_query_ctx()
        mirror = co.collide_f32(d.states, d.headings, f[8:].reshape(16, 4), int(i[5]), f[2:8], i[0:2],
                                corridor[0], hl, hw, rc2)
        valid = (d.flags & 1) != 0
        stats["valid"] += int(valid.sum())
        stats["collide"] += int((mirror[valid] != 0).sum())
        stats["mirror_mismatch"] += int((mirror[valid] != (d.flags[valid] & 6)).sum())
    goals = np.array([[1.0, 0.2, 0.1], [2.5, -0.8, -0.4], [3.5, 1.2, 0.6], [0.8, 0.0, 0.0], [2.0, 0.6, 0.9]])
    states, params, ok = eng.generate(goals)
    assert ok.any()
    for g, s in zip(goals[ok], states[ok]):
        ref = co.spiral(g, n_newton=12, m=M)[1]
        assert H.close(s, ref, scale=H.traj_scale(ref)).all(), (M, g, np.abs(s - ref).max(axis=0))
    H.record_parity("eval_instances_reference_m%d" % M, stats)
    assert stats["mirror_mismatch"] == 0, stats
    if M >= 4:   # two or three samples leave most candidates invalid, on the oracle's side too
        assert stats["valid"] >= 40 and stats["both_valid"] >= 20, stats


@pytest.mark.parametrize("M", MS)
def test_regimes(ellipse, corridor, M):
    """every reachable regime of M's bucket bit for bit against single queries, the PW twin of
    every batch regime, dense lone queries against their shards; every built instance of the
    bucket runs"""
    eng, cfg, world = _engine(ellipse, corridor, M, 28, kappa_max=3.0)
    sm = _sm(eng)
    stats, ran = {}, set()
    row = _row(M)
    regimes = _workloads(M, sm)
    for inst, wls in regimes.items():
        for n, S, lone in wls:
            name = "nw%d_minb%d_wide%d_n%d_s%d%s" % (inst[1], inst[2], inst[3], n, S, "_lone" if lone else "")
            if lone and eval_choice(n, S, M, 0, lone, False, sm)["persistent"]:
                _dense_regime(eng, ellipse, M, sm, n, 4000 + n, stats, name)
                ran.add(stats[name]["instance"])
            else:
                # (a lone query on a static grid plans as a batch of one scenario)
                ran |= set(_batch_regime(eng, ellipse, M, sm, n, S, 5000 + n + S, stats, name))
    if row["nw4"]:
        # ragged chunks of the throughput regime: groups of four with idle members
        S = 8 * row["nw4"] * sm
        for n in RAGGED:
            assert eval_choice(n, S, M, 0, False, False, sm)["nw"] == 4
            ran |= set(_batch_regime(eng, ellipse, M, sm, n, S, 6000 + n, stats, "throughput_n%d" % n))
    for S in SAMPLER:
        ran |= set(_batch_regime(eng, ellipse, M, sm, 28, S, 7000 + S, stats, "sampler_s%d" % S))
    # every built instance of the bucket ran
    names = set()
    for nw in (4, 7, 8):
        if row["nw%d" % nw]:
            names |= {"eval_kernel<%d,%d,%d,%d,%d,%s>" % (row["ipl"], row["s"], row["sg"], nw, row["nw%d" % nw], pw)
                      for pw in ("false", "true")}
    if row["wide"]:
        names.add("eval_kernel<%d,%d,%d,8,%d,false>" % (row["ipl"], row["s"], row["sg"], row["wide"]))
    ran = {r.replace(" persistent", "") for r in ran}
    stats["instances"] = sorted(ran)
    H.record_parity("eval_instances_regimes_m%d" % M, stats)
    assert names <= ran, (sorted(names - ran), sorted(ran))


@pytest.mark.parametrize("M", ONCE)
def test_bucket_options(ellipse, corridor, M):
    """once per bucket: the pruned window scan, the G1-clothoid generator and disc collisions on
    each batch regime against the default path and single queries, and the dense lone regimes
    against oracle slices"""
    eng, cfg, world = _engine(ellipse, corridor, M, 28, kappa_max=3.0, window=256)
    sm = _sm(eng)
    stats = {}
    regimes = _workloads(M, sm)
    for inst, wls in regimes.items():
        for n, S, lone in wls:
            if lone:
                continue
            la, wd = _grid(n)
            eng.set_goal_grid(la, wd)
            poses, opp, n_opp = synth.scenario_batch(ellipse, S, K_OPP, 8000 + n + S)
            # without per-term costs the pruned scan also skips colliding candidates
            for terms in (True, False):
                full = _batch_dev(eng, poses, opp, n_opp, want_terms=terms)
                eng.configure(prune_window=1)
                pr = _batch_dev(eng, poses, opp, n_opp, want_terms=terms)
                _confirm(eng, n, S, M, sm)
                eng.configure(prune_window=0)
                fields = FIELDS if terms else tuple(k for k in FIELDS if k != "terms")
                diff = [k for k in fields if not np.array_equal(getattr(pr, k), getattr(full, k))]
                assert not diff, ("prune", n, S, terms, diff)
            idx = np.sort(np.random.default_rng(n + S).choice(S, min(S, 16), replace=False))
            for opt in (dict(generator=1), dict(collision_mode=1)):
                eng.configure(**opt)
                b = _batch_dev(eng, poses, opp, n_opp)
                bad = _single_mismatches(eng, b, poses, opp, n_opp, idx)
                assert not bad, (opt, n, S, bad)
                eng.configure(generator=0, collision_mode=0)
            stats["batch_n%d_s%d" % (n, S)] = {"prune_gen1_disc": "ok", "singles": len(idx)}
    # the G1 generator and disc collisions against the oracle on single queries
    eng.set_goal_grid(*_grid(28))
    for opt in (dict(generator=1), dict(collision_mode=1)):
        eng.configure(**opt)
        ocfg = H.oracle_config_from_engine(eng)
        for seed in (8200 + M, 8300 + M):
            pose, opp1 = H.scenario(ellipse, seed, K_OPP)
            d = eng.plan(pose, opp1, update_prev=False, want_states=True, want_map=True)
            H.compare_plan(d, co.plan(ocfg, world, pose, opp1, want_states=True), ocfg)
        eng.configure(generator=0, collision_mode=0)
    # the dense lone regimes against oracle slices of 512 candidates
    eng.configure(window=128)
    ocfg = H.oracle_config_from_engine(eng)
    for inst, wls in regimes.items():
        for n, S, lone in wls:
            if not lone:
                continue
            pose, opp1, whole = _dense_regime(eng, ellipse, M, sm, n, 8400 + n, stats, "dense_n%d" % n)
            w = _world(eng, ellipse, corridor, n)
            counts = {}
            for lo in (0, n // 2 - 256, n - 512):
                _oracle_slice(ocfg, w, pose, opp1, whole.costs, whole.flags, lo, lo + 512, counts)
            stats["dense_oracle_n%d" % n] = counts
            assert counts["finite"] > 0, counts
    H.record_parity("eval_instances_options_m%d" % M, stats)


@pytest.mark.parametrize("M", ONCE)
def test_window_limit(corridor, M):
    """the largest window of every reachable instance runs and matches the oracle; one padded
    step more is F1L_ERR_TOO_LARGE and leaves the handle working"""
    track = synth.ellipse_track(n=8000)
    eng, cfg, world = _engine(track, corridor, M, 28, kappa_max=3.0)
    sm = _sm(eng)
    stats = {}
    # per instance the workload with the most candidates: the most finite costs to compare
    pick = {}
    for wls in _workloads(M, sm).values():
        for n, S, lone in wls:
            for pw in ((False,) if lone else (False, True)):
                key = instance(eval_choice(n, S, M, 0, lone, pw, sm))
                if key not in pick or n * S > pick[key][0] * pick[key][1]:
                    pick[key] = (n, S, lone, pw)
    for key, (n, S, lone, pw) in sorted(pick.items()):
        wmax = eval_choice(n, S, M, 0, lone, pw, sm)["max_window"]
        assert wmax < track.shape[0] - 1
        la, wd = _grid(n)
        eng.set_goal_grid(la, wd)
        eng.configure(window=wmax)
        ocfg = H.oracle_config_from_engine(eng)
        w = _world(eng, track, corridor, n)
        poses, opp, n_opp = synth.scenario_batch(track, S, K_OPP, 9000 + n + S)
        n_opp[:] = 0   # no opponents: more finite costs to compare
        W = np.tile(np.array(list(eng.config.weights), np.float32), (S, 1)) if pw else None

        def run():
            if lone:
                d = eng.plan(poses[0], None, update_prev=False)
                return d.costs[None], d.flags[None]
            b = _batch_dev(eng, poses, opp, n_opp, weights=W)
            return b.costs, b.flags
        costs, flags = run()
        got = _confirm(eng, n, S, M, sm, lone, pw)
        # up to four scenarios with finite costs, each on a slice of 64 candidates from its first
        # finite one
        counts = {}
        fin = np.nonzero(np.isfinite(costs).any(axis=1))[0]
        for s in fin[np.linspace(0, fin.size - 1, min(4, fin.size)).astype(int)] if fin.size else []:
            lo = min(int(np.argmax(np.isfinite(costs[s]))), max(n - 64, 0))
            _oracle_slice(ocfg, w, poses[s], None, costs[s], flags[s], lo, min(n, lo + 64), counts)
        eng.configure(window=wmax + 1)
        with pytest.raises(F1LError, match="error -5"):
            run()
        eng.configure(window=wmax)
        again = run()
        assert np.array_equal(again[0], costs) and np.array_equal(again[1], flags)
        stats[got["name"]] = dict(window=wmax, n_cand=n, S=S, **counts)
        assert counts.get("finite", 0) > 0, (got["name"], stats[got["name"]])
    H.record_parity("eval_instances_window_m%d" % M, stats)
    row = _row(M)
    built = sum(2 for nw in (4, 7, 8) if row["nw%d" % nw]) + (1 if row["wide"] else 0)
    assert len(pick) == built, sorted(pick)
    assert sum(v["finite"] for v in stats.values()) >= 50, stats
