"""bench.py --dump-outputs: every output of the timed step, float32 / float64 and finite only
(non-finite entries masked), within the size budget, the same seeded rows from run to run.  CPU
tensors stand in for the device buffers."""
import os
import types

import numpy as np
import torch

import bench


def _arm(S, C, M):
    """random outputs with what the planner returns beside plain values: +inf costs (invalid or
    collided candidates), +inf best_cost (no feasible candidate), a non-finite trajectory"""
    g = torch.Generator().manual_seed(3)
    arm = types.SimpleNamespace(
        S=S, o_idx=torch.randint(0, C, (S,), dtype=torch.int32, generator=g),
        o_cost=torch.rand(S, generator=g), o_traj=torch.rand(S, M, 4, generator=g),
        o_costs=torch.rand(S, C, generator=g),
        o_flags=torch.randint(0, 256, (S, C), dtype=torch.int32, generator=g).to(torch.uint8),
        o_ss=torch.rand(S, 2, dtype=torch.float64, generator=g))
    arm.o_costs[torch.rand(S, C, generator=g) < 0.15] = float("inf")
    arm.o_cost[::7] = float("inf")
    arm.o_traj[::5, 3, 1] = float("nan")
    arm.o_ss[::11, 0] = float("nan")
    return arm


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _unmask(out, name):
    """the written values, NaN where <name>_finite marks a non-finite entry (written as 0)"""
    v, ok = out[name], out[name + "_finite"]
    assert set(np.unique(ok)) <= {0.0, 1.0} and not v[ok == 0].any()
    return np.where(ok == 1, v, np.nan)


def _same(a, b):
    """equal, with every non-finite entry of b (inf or nan) masked in a"""
    return np.array_equal(np.isfinite(a), np.isfinite(b)) and np.array_equal(a[np.isfinite(a)], b[np.isfinite(b)])


def _check(arm, out):
    assert set(out) == {"scenarios", "best_idx", "best_cost", "best_cost_finite", "costs", "costs_finite",
                        "flags", "steer_speed", "steer_speed_finite", "best_traj_scenarios", "best_traj",
                        "best_traj_finite"}
    assert all(v.dtype in (np.float32, np.float64) for v in out.values())
    assert all(np.isfinite(v).all() for v in out.values())
    r = out["scenarios"].astype(np.int64)
    t = out["best_traj_scenarios"].astype(np.int64)
    assert np.array_equal(out["best_idx"], arm.o_idx.numpy()[r])
    assert np.array_equal(out["flags"], arm.o_flags.numpy()[r])
    assert _same(_unmask(out, "best_cost"), arm.o_cost.numpy()[r])
    assert _same(_unmask(out, "costs"), arm.o_costs.numpy()[r])
    assert _same(_unmask(out, "steer_speed"), arm.o_ss.numpy()[r])
    traj = arm.o_traj.numpy()[t]
    ok = np.isfinite(traj).all(axis=(1, 2))
    assert np.array_equal(out["best_traj_finite"], ok) and not ok.all()
    assert np.array_equal(out["best_traj"][ok], traj[ok])
    assert not out["best_traj"][~ok][~np.isfinite(traj[~ok])].any()
    return r, t


def test_small_batch_is_written_whole(tmp_path):
    arm = _arm(300, 28, 100)
    bench.dump_outputs(torch, arm, str(tmp_path))
    r, t = _check(arm, _load(str(tmp_path)))
    assert np.array_equal(r, np.arange(300)) and np.array_equal(t, np.arange(300))


def test_large_batch_is_a_seeded_sample_within_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 400_000)
    arm = _arm(3000, 28, 100)
    bench.dump_outputs(torch, arm, str(tmp_path / "a"))
    bench.dump_outputs(torch, arm, str(tmp_path / "b"))
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    r, t = _check(arm, a)
    assert 0 < len(t) < len(r) < 3000 and len(np.unique(r)) == len(r)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.nbytes for v in a.values()) <= 400_000


def test_default_workload_fits_64_mb(tmp_path):
    """the bench's own shape (10^5 scenarios x 4x7 goals, M = 100): every scenario of the
    per-candidate outputs, a sample of the trajectories, 64 MB on disk at most"""
    arm = _arm(bench.S_PER_GPU, 28, bench.PLAN_CFG["n_samples"])
    bench.dump_outputs(torch, arm, str(tmp_path))
    r, t = _check(arm, _load(str(tmp_path)))
    assert len(r) == bench.S_PER_GPU and len(t) > 10000
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)) <= 64 * 10**6
