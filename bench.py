#!/usr/bin/env python
"""bench.py -- lattice candidates evaluated / s (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c4]
                    [--dump-outputs DIR]

A step = one pass of the hot path (sampler -> spiral generation -> fused cost + collision ->
argmin -> tracker) over one batch of synthetic planning scenarios (SURVEY.md 8d, config 4):
per GPU 10^5 independent scenarios x the default 4x7 goal grid = 2.8e6 candidates, M=100 arc
samples, raceline window W=128, up to 8 opponents, occupancy grid on.  Scenarios are independent,
so ranks shard them with no data-path collective (weak scaling; the only collectives are the
barrier and the max-over-ranks of the step time).

`value` is device-resident throughput (inputs in HBM, CUDA events); `e2e` is the same metric
through the public Python API (LatticePlanner.plan_batch) with pinned HOST buffers, H2D and D2H
inside the timed region.  `--impl reference` times the CPU oracle port (the reference's lattice
path cannot execute: SURVEY.md section 0) on all host cores on a bounded sample of the workload.

`--dump-outputs DIR` writes what the last timed step of the device-resident arm returned (rank 0)
as DIR/<name>.npy (dump_outputs).  The scenarios are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from f1tenth_planning_b200 import flops as F  # noqa: E402
from f1tenth_planning_b200 import synth  # noqa: E402

METRIC = "lattice candidates evaluated/sec"
UNIT = "candidates/s"
S_PER_GPU = 100000
K_OPP = 8
PLAN_CFG = dict(n_samples=100, n_newton=8, window=128, kappa_max=0.0)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c4"])
    ap.add_argument("--scenarios", type=int, default=S_PER_GPU, help="scenarios per GPU per step")
    ap.add_argument("--prune", type=int, default=0, choices=[0, 1],
                    help="prune_window of the headline run (0: every sample against all W window "
                         "segments, the SURVEY FLOP model; 1: provably-far segments skipped)")
    ap.add_argument("--no-extras", action="store_true", help="skip the C2/C3/C5 side measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true",
                    help="kernel A/B runs: device-resident arm only, prints a short JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """rows seen so far (call at the start of the timed region; the sampler itself is started
        earlier because nvidia-smi needs ~0.2 s before its first row)"""
        self.first = len(self.rows)

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

    def window(self):
        """clocks / throttle reasons of the rows since mark() (the sampler keeps running)"""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        last = len(self.rows)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows[getattr(self, "first", 0):last] or self.rows[-3:]
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for n, v in zip(names, p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


PROFILE_MD = "profiles/r2_eval_kernel.md" if os.path.exists(os.path.join(ROOT, "profiles", "r2_eval_kernel.md")) \
    else "profiles/r1_eval_kernel.md"


def profiled_dram_bytes(path=None):
    """dram__bytes_read.sum + dram__bytes_write.sum of one eval_kernel launch of the bench workload,
    from the committed ncu --set full summary (bench.py cannot run under ncu itself)."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, seen = 0.0, 0
    path = path or os.path.join(ROOT, PROFILE_MD)
    try:
        for ln in open(path):
            c = [x.strip() for x in ln.split("|")]
            if len(c) > 3 and c[1] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tot += float(c[2]) * unit[c[3]]
                seen += 1
    except Exception:
        return None
    return int(tot) if seen == 2 else None


def workload(seed_rank, S):
    """Scenario set of rank `seed_rank`: always drawn as the full S_PER_GPU-scenario batch of that
    seed and then cut to its first S, so every arm (device-resident, end to end, CPU baseline,
    --impl reference, strong-scaling shards) sees a prefix / slice of the SAME scenarios (the
    generator's stream depends on the batch size)."""
    track = synth.ellipse_track()
    grid = synth.corridor_grid()
    la, wd = synth.goal_grid(4)
    poses, opp, n_opp = synth.scenario_batch(track, max(S, S_PER_GPU), K_OPP, 1004 + 7919 * seed_rank)
    return track, grid, la, wd, poses[:S].copy(), opp[:S].copy(), n_opp[:S].copy()


def work_flops(flags, M, seg_steps, n_opp_mean):
    """algorithmic FLOPs of one step (appendix D) from the flags it produced and the kernel's own
    work counter: a candidate that failed validation stops after generation; the Newton term counts
    the quadrature passes the candidate actually used (flag bits 4..7) instead of the nominal 8;
    the deviation term is 17 M per (candidate, window segment) pair the kernel actually tested
    (`seg_steps`, f1l_get_stats) -- W = 128 for every valid candidate in the headline run, fewer
    with prune_window = 1, which also drops the pass for collided candidates."""
    valid = (flags & 1) != 0
    passes = (flags >> 4).astype(np.float64)
    n_full = int(valid.sum())
    n_short = int(valid.size - n_full)
    base = (n_full * F.candidate_flops(M=M, W=0, K=n_opp_mean, I=0, full=True) +
            n_short * F.candidate_flops(M=M, W=0, K=n_opp_mean, I=0, full=False))
    newton = float(passes.sum()) * (44 * (F.Q_NEWTON + 1) + 110)
    return base + 17.0 * M * float(seg_steps) + newton, n_full / valid.size, float(passes.mean())


# ------------------------------------------------------------------------------------------------
def host_threads():
    """all host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle's
    OpenMP loops take an explicit num_threads, so that default does not apply)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_reference_rate(track, grid, la, wd, poses, opp, n_opp, seconds, threads=None):
    """oracle port on the host cores: (cand/s, sample size, threads)"""
    from oracle import c_oracle as co
    threads = threads or host_threads()
    world = co.World_(track, la, wd, grid=grid[0], grid_origin=grid[1], grid_res=grid[2])
    cfg = co.default_config(**PLAN_CFG)
    C = world.n_candidates
    n0 = min(poses.shape[0], 16 * threads)
    t = time.perf_counter()
    co.plan_batch(cfg, world, poses[:n0], opp[:n0], n_opp[:n0], n_threads=threads,
                  want_traj=True, want_costs=True)
    rate = n0 * C / (time.perf_counter() - t)
    n = int(max(n0, min(poses.shape[0], rate * seconds / C)))
    t = time.perf_counter()
    co.plan_batch(cfg, world, poses[:n], opp[:n], n_opp[:n], n_threads=threads, want_traj=True,
                  want_costs=True)
    dt = time.perf_counter() - t
    return n * C / dt, n, threads, dt


def run_reference(args):
    """--impl reference: the CPU path on the host cores, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import c_oracle as co
    threads = host_threads()
    track, grid, la, wd, poses, opp, n_opp = workload(0, S_PER_GPU)   # the GPU arm's rank-0 scenarios
    world = co.World_(track, la, wd, grid=grid[0], grid_origin=grid[1], grid_res=grid[2])
    cfg = co.default_config(**PLAN_CFG)
    C = world.n_candidates
    # size one step so that warmup + steps fit in ~2 minutes
    n0 = 16 * threads
    t = time.perf_counter()
    co.plan_batch(cfg, world, poses[:n0], opp[:n0], n_opp[:n0], n_threads=threads)
    rate = n0 * C / (time.perf_counter() - t)
    budget = min(10.0, 120.0 / max(1, args.steps + args.warmup))
    n = int(max(n0, min(poses.shape[0], rate * budget / C)))
    for _ in range(args.warmup):
        co.plan_batch(cfg, world, poses[:n], opp[:n], n_opp[:n], n_threads=threads)
    t = time.perf_counter()
    for _ in range(args.steps):
        co.plan_batch(cfg, world, poses[:n], opp[:n], n_opp[:n], n_threads=threads)
    dt = time.perf_counter() - t
    value = n * C * args.steps / dt
    sample = ("the first %d of the GPU arm's %d scenarios x %d candidates per step (bounded sample of the "
              "same workload, same seed)" % (n, S_PER_GPU, C))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "c4: independent scenarios x 4x7 goal grid, M=100, W=128, <=8 opponents, grid on",
                   "note": "reference lattice path cannot execute (SURVEY 0.1); this is the C oracle port "
                           "(oracle/c/f1o.c), OpenMP over scenarios"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def extras(track, grid, device, fp32_peak=None):
    """side measurements (not the headline): C3 plan() latency, C2 poses/s, C5 dense sweep."""
    import torch
    from f1tenth_planning_b200.engine import Engine
    out = {}
    # C1: the reference's own case -- LatticePlanner.plan(), default 4x7 grid, one opponent --
    # through the public class, next to the CPU oracle's plan() of the same queries
    from f1tenth_planning_b200 import LatticePlanner
    from oracle import c_oracle as co
    la1, wd1 = synth.goal_grid(1)
    pl = LatticePlanner(waypoints=track, device=device, n_samples=100, window=128)
    pl.set_map(*grid)
    p1, o1, _ = synth.scenario_batch(track, 64, 1, 1001)
    for i in range(5):
        pl.plan(*p1[i], opponent_poses=o1[i])
    ts = []
    for i in range(1000):
        t = time.perf_counter()
        pl.plan(*p1[i % 64], opponent_poses=o1[i % 64])
        ts.append(time.perf_counter() - t)
    out["c1_plan_p50_us"] = 1e6 * float(np.percentile(ts, 50))
    out["c1_plan_p99_us"] = 1e6 * float(np.percentile(ts, 99))
    ocfg = co.default_config(n_samples=100, window=128)
    world = co.World_(track, la1, wd1, grid=grid[0], grid_origin=grid[1], grid_res=grid[2])
    ts = []
    for i in range(40):
        t = time.perf_counter()
        co.plan(ocfg, world, p1[i % 64], o1[i % 64])
        ts.append(time.perf_counter() - t)
    out["c1_cpu_oracle_plan_p50_us"] = 1e6 * float(np.percentile(ts, 50))
    # C3: single query, 4096 candidates
    la, wd = synth.goal_grid(3)
    eng = Engine(device=device, n_samples=100, window=128)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    poses, opp, n_opp = synth.scenario_batch(track, 64, 8, 1003)
    for i in range(5):
        eng.plan(poses[i], opp[i], update_prev=False, detail=False)
    ts = []
    for i in range(300):
        s = i % 64
        t = time.perf_counter()
        eng.plan(poses[s], opp[s], update_prev=True, detail=False)
        ts.append(time.perf_counter() - t)
    out["c3_plan_p50_us"] = 1e6 * float(np.percentile(ts, 50))
    out["c3_plan_p99_us"] = 1e6 * float(np.percentile(ts, 99))
    eng.set_timing(True)
    for i in range(20):
        eng.plan(poses[i], opp[i], update_prev=False, detail=False)
    sm, ev, se, n = eng.mean_kernel_ms()
    out["c3_kernel_us"] = {"sample": 1e3 * sm, "eval": 1e3 * ev, "select": 1e3 * se}
    out["c3_eval_candidates_per_s"] = 4096 / (ev * 1e-3) if ev > 0 else None
    eng.close()
    # the CPU oracle's plan() of the same C3 queries (one core: a single query is sequential)
    ocfg3 = co.default_config(n_samples=100, window=128)
    world3 = co.World_(track, la, wd, grid=grid[0], grid_origin=grid[1], grid_res=grid[2])
    ts = []
    for i in range(3):
        t = time.perf_counter()
        co.plan(ocfg3, world3, poses[i], opp[i, :n_opp[i]])
        ts.append(time.perf_counter() - t)
    out["c3_cpu_oracle_plan_p50_us"] = 1e6 * float(np.percentile(ts, 50))
    out["c3_cpu_oracle_cores"] = 1
    # C5: dense sweep 65536 x 200
    la, wd = synth.goal_grid(5)
    eng = Engine(device=device, n_samples=200, window=128)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    eng.set_timing(True)
    for i in range(3):
        eng.plan(poses[i], opp[i], update_prev=False, detail=False)
    eng.set_timing(True)
    ts = []
    for i in range(10):
        t = time.perf_counter()
        eng.plan(poses[i], opp[i], update_prev=False, detail=False)
        ts.append(time.perf_counter() - t)
    sm, ev, se, n = eng.mean_kernel_ms()
    out["c5_plan_p50_us"] = 1e6 * float(np.percentile(ts, 50))
    out["c5_eval_candidates_per_s"] = 65536 / (ev * 1e-3) if ev > 0 else None
    eng.close()
    # CPU oracle on a bounded slice of the same C5 query (2048 of the 65536 candidates, one core),
    # and the whole query extrapolated linearly from it
    ocfg5 = co.default_config(n_samples=200, window=128)
    world5 = co.World_(track, la, wd, grid=grid[0], grid_origin=grid[1], grid_res=grid[2])
    t = time.perf_counter()
    co.plan(ocfg5, world5, poses[0], opp[0, :n_opp[0]], c_begin=32768, c_end=32768 + 2048)
    dt = time.perf_counter() - t
    out["c5_cpu_oracle_candidates_per_s"] = 2048 / dt
    out["c5_cpu_oracle_plan_extrapolated_us"] = 1e6 * dt * 65536 / 2048
    out["c5_cpu_oracle_cores"] = 1
    out["c5_cpu_oracle_sample"] = "candidates [32768, 34816) of query 0, %.2f s" % dt
    # C2: 10^5 poses pure pursuit, device resident
    eng = Engine(device=device)
    eng.set_track(track)
    rng = np.random.default_rng(1002)
    pp, _ = synth.random_poses(track, 100000, rng)
    dev = torch.device("cuda", device)
    tp = torch.from_numpy(np.ascontiguousarray(pp[:, :3])).to(dev)
    near = torch.empty(100000, 4, dtype=torch.float64, device=dev)
    ni = torch.empty(100000, dtype=torch.int32, device=dev)
    look = torch.empty(100000, 4, dtype=torch.float64, device=dev)
    li = torch.empty(100000, dtype=torch.int32, device=dev)
    act = torch.empty(100000, 2, dtype=torch.float64, device=dev)
    stt = torch.empty(100000, dtype=torch.int32, device=dev)
    for _ in range(3):
        eng.pure_pursuit_batch_dev(tp, 0.8, near, ni, look, li, act, stt)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        eng.pure_pursuit_batch_dev(tp, 0.8, near, ni, look, li, act, stt)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / 10
    out["c2_poses_per_s"] = 100000 / (ms * 1e-3)
    out["c2_ms"] = ms
    out["c2_fp32_tflops"] = 100000 * F.pose_flops(track.shape[0]) / (ms * 1e-3) / 1e12
    # K1's own roofline object: F_pose = 17 (N - 1) + 60 FLOP (SURVEY 8d) x 10^5 poses per launch pair
    out["c2_roofline"] = {"bound": "fp32", "achieved": out["c2_fp32_tflops"], "peak": fp32_peak,
                          "unit": "TFLOP/s", "frac": out["c2_fp32_tflops"] / fp32_peak if fp32_peak else None,
                          "kernel": "pp_scan_kernel + pp_finish_kernel", "ms": ms,
                          "flops_per_launch": 100000 * F.pose_flops(track.shape[0])}
    eng.close()
    # CPU oracle (pinned to the reference's nearest_point / pure pursuit) on a bounded sample of
    # the same poses: one core -- the reference is single-threaded -- and all host cores
    th = host_threads()
    for key, nt, n in (("c2_cpu_oracle_poses_per_s_1core", 1, 4000), ("c2_cpu_oracle_poses_per_s_all_cores", th, 4000 * th)):
        n = min(n, 100000)
        t = time.perf_counter()
        co.pure_pursuit_batch(track, pp[:n, :3], 0.8, n_threads=nt)
        out[key] = n / (time.perf_counter() - t)
    out["c2_cpu_oracle_cores"] = th
    return out


def sharded_dense_query(track, grid, device, rank, world_size, dev):
    """config 5 across ranks: every rank evaluates a contiguous block of the 65536 candidates of
    ONE query (f1l_plan_shard) and the ranks' (cost, idx) minima are exchanged (SURVEY 8e) --
    (a) inside the select kernel through peer memory over NVLink (Engine.attach_peers; every
    rank's plan() returns the global winner), (b) for comparison by a 16-byte NCCL all-gather plus
    a host min (sharding.reduce_best).  Latency = barrier-to-result on the slowest rank."""
    import torch
    import torch.distributed as dist
    from f1tenth_planning_b200 import sharding
    from f1tenth_planning_b200.engine import Engine
    la, wd = synth.goal_grid(5)
    eng = Engine(device=device, n_samples=200, window=128)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    C = eng.n_candidates
    lo, hi = sharding.block(C, rank, world_size)
    poses, opp, n_opp = synth.scenario_batch(track, 16, 8, 1005)   # same on every rank

    start = torch.zeros(1, dtype=torch.float64, device=dev)

    def run(n_rep, reduce_on_host, by_rows):
        """Every rank starts query i at the same instant: rank 0 broadcasts a start time 2 ms
        ahead on the host's monotonic clock (time.perf_counter is CLOCK_MONOTONIC, shared by the
        processes of one node) and the ranks spin until it comes -- a barrier's exit skew
        (~100 us between ranks) would otherwise be charged to the query.  Latency of a query =
        the latest finish over the ranks minus that common start."""
        ts, tp, bests = [], [], []
        for i in range(3 + n_rep):
            s = i % 16
            torch.cuda.synchronize(dev)
            dist.barrier()
            if rank == 0:
                start[0] = time.perf_counter() + 2e-3
            dist.broadcast(start, 0)
            t0 = float(start.item())
            while time.perf_counter() < t0:
                pass
            if by_rows:
                d = eng.plan(poses[s], opp[s], update_prev=False, detail=False, rows=(rank, world_size))
            else:
                d = eng.plan(poses[s], opp[s], update_prev=False, detail=False, shard=(lo, hi))
            t1 = time.perf_counter()
            best = (sharding.reduce_best(d.best_cost, d.best_idx) if reduce_on_host
                    else (float(d.best_cost), int(d.best_idx)))
            dt = time.perf_counter() - t0
            if i >= 3:
                ts.append(dt)
                tp.append(t1 - t0)
                bests.append((float(np.float32(best[0])), int(best[1])))
        t = torch.tensor(ts, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy(), np.array(tp), bests

    ts_n, tp_n, best_n = run(32, True, False)   # (b) contiguous blocks, NCCL all-gather + host min
    _, tp_r, _ = run(32, True, True)            # local time of a row-interleaved shard
    eng.attach_peers()
    ts_c, _, best_c = run(32, False, False)     # peer memory, contiguous blocks
    ts_p, _, best_p = run(32, False, True)      # (a) peer memory, row-interleaved shards
    # the same query with prune_window = 1: window segments that provably cannot be nearest to any
    # sample of a candidate are skipped; costs, hence the winner, are bit-identical
    eng.configure(prune_window=1)
    ts_q, _, best_q = run(32, False, True)
    eng.configure(prune_window=0)
    eng.detach_peers()
    # where a rank's local time goes: device time of its three kernels (plain launches, CUDA events)
    eng.set_timing(True)
    for i in range(24):
        eng.plan(poses[i % 16], opp[i % 16], update_prev=False, detail=False, rows=(rank, world_size))
    k_ms = eng.mean_kernel_ms()[:3]
    eng.set_timing(False)
    tk = torch.tensor(k_ms, dtype=torch.float64, device=dev)
    dist.all_reduce(tk, op=dist.ReduceOp.MAX)
    k_us = [1e3 * float(v) for v in tk.cpu().numpy()]
    eng.close()
    tl = torch.tensor([np.percentile(tp_n, 50), np.percentile(tp_r, 50)], dtype=torch.float64, device=dev)
    dist.all_reduce(tl, op=dist.ReduceOp.MAX)   # the slowest rank's local plan
    tl = tl.cpu().numpy()
    return {"c5_sharded_plan_p50_us": 1e6 * float(np.percentile(ts_p, 50)),
            "c5_sharded_plan_p99_us": 1e6 * float(np.percentile(ts_p, 99)),
            "c5_sharded_candidates_per_s": C / float(np.percentile(ts_p, 50)),
            "c5_sharded_exchange": "row-interleaved shards (f1l_plan_rows), each rank samples only its rows; "
                                   "(key, goal centre) entries exchanged over peer memory (CUDA IPC over "
                                   "NVLink, system-scope stores + arrival counters inside select_kernel)",
            "c5_sharded_blocks_peer_p50_us": 1e6 * float(np.percentile(ts_c, 50)),
            "c5_sharded_blocks_nccl_gather_p50_us": 1e6 * float(np.percentile(ts_n, 50)),
            "c5_sharded_local_plan_p50_us": {"rows_slowest_rank": 1e6 * float(tl[1]),
                                             "blocks_slowest_rank": 1e6 * float(tl[0])},
            "c5_sharded_pruned_plan_p50_us": 1e6 * float(np.percentile(ts_q, 50)),
            "c5_sharded_pruned_note": "prune_window=1: provably-irrelevant window segments skipped, "
                                      "bit-identical costs and winner (c5_sharded_paths_agree covers it)",
            "c5_sharded_kernel_us_slowest_rank": {"sample": k_us[0], "eval": k_us[1], "select": k_us[2]},
            "c5_sharded_paths_agree": best_n == best_p and best_c == best_p and best_q == best_p,
            "c5_candidates_per_rank": hi - lo, "c5_last_best": list(best_p[-1])}


class DeviceArm:
    """device-resident inputs / outputs of one rank for S scenarios"""

    def __init__(self, torch, dev, eng, poses, opp, n_opp):
        S, C, M = poses.shape[0], eng.n_candidates, eng.n_samples
        self.eng, self.S = eng, S
        self.tp = torch.from_numpy(poses).to(dev)
        self.to = torch.from_numpy(opp).to(dev)
        self.tn = torch.from_numpy(n_opp).to(dev)
        self.o_idx = torch.empty(S, dtype=torch.int32, device=dev)
        self.o_cost = torch.empty(S, dtype=torch.float32, device=dev)
        self.o_traj = torch.empty(S, M, 4, dtype=torch.float32, device=dev)
        self.o_costs = torch.empty(S, C, dtype=torch.float32, device=dev)
        self.o_flags = torch.empty(S, C, dtype=torch.uint8, device=dev)
        self.o_ss = torch.empty(S, 2, dtype=torch.float64, device=dev)

    def step(self):
        self.eng.plan_batch_dev(self.tp, self.to, self.tn, best_idx=self.o_idx, best_cost=self.o_cost,
                                best_traj=self.o_traj, costs=self.o_costs, flags=self.o_flags,
                                steer_speed=self.o_ss)


DUMP_BYTES = 60 * 10**6   # with the .npy headers and file-system blocks, under 64 MB


def dump_outputs(torch, arm, out_dir):
    """Every output of DeviceArm.step() as out_dir/<name>.npy in float32 / float64 (indices and
    flags converted exactly), DUMP_BYTES in all.  Every value written is finite: a non-finite
    entry (the +inf cost of an invalid or collided candidate, the +inf best_cost of a scenario
    without a feasible candidate) is written as 0, and <name>_finite.npy holds 1 where the value
    is finite (per scenario for best_traj).  The per-scenario outputs cover every scenario while
    they fit in 2/3 of the budget (the default size does), else a seeded sample of scenarios;
    best_traj [S, M, 4] (160 MB at the default size) a seeded sample in the rest.  scenarios.npy
    and best_traj_scenarios.npy give the scenario index of each row."""
    S, M, C = arm.S, arm.o_traj.shape[1], arm.o_costs.shape[1]
    rng = np.random.default_rng(0)

    def rows(budget, row_bytes):
        n = max(0, budget // row_bytes)
        return np.arange(S) if n >= S else np.sort(rng.choice(S, n, replace=False))

    def finite(v, per_scenario):
        ok = torch.isfinite(v)
        return torch.where(ok, v, torch.zeros_like(v)), (ok.flatten(1).all(1) if per_scenario else ok).float()

    # index, best_idx, best_cost + mask, costs + mask, flags, steer_speed + mask
    row_bytes = 8 + 8 + 8 + C * 12 + 24
    r = rows(DUMP_BYTES * 2 // 3, row_bytes)
    t = rows(DUMP_BYTES - len(r) * row_bytes - (16 << 10), 8 + M * 16 + 4)   # 16 KB: .npy headers
    ri = torch.from_numpy(r).to(arm.o_costs.device)
    ti = torch.from_numpy(t).to(arm.o_costs.device)
    out = {"scenarios": r.astype(np.float64), "best_idx": arm.o_idx[ri].double(),
           "flags": arm.o_flags[ri].float(), "best_traj_scenarios": t.astype(np.float64)}
    for name, v, per_scenario in (("best_cost", arm.o_cost[ri], False), ("costs", arm.o_costs[ri], False),
                                  ("steer_speed", arm.o_ss[ri], False), ("best_traj", arm.o_traj[ti], True)):
        out[name], out[name + "_finite"] = finite(v, per_scenario)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy() if torch.is_tensor(v) else v)


class HostArm:
    """the public API with pinned HOST buffers: every output the device-resident arm writes"""

    def __init__(self, planner, pinned_empty, poses, opp, n_opp):
        S, C, M = poses.shape[0], planner.engine.n_candidates, planner.engine.n_samples
        self.planner = planner
        self.h_poses = pinned_empty(poses.shape, np.float64); self.h_poses[:] = poses
        self.h_opp = pinned_empty(opp.shape, np.float64); self.h_opp[:] = opp
        self.h_nopp = pinned_empty(n_opp.shape, np.int32); self.h_nopp[:] = n_opp
        self.h_out = {"best_idx": pinned_empty((S,), np.int32), "best_cost": pinned_empty((S,), np.float32),
                      "best_traj": pinned_empty((S, M, 4), np.float32),
                      "costs": pinned_empty((S, C), np.float32), "flags": pinned_empty((S, C), np.uint8),
                      "steer_speed": pinned_empty((S, 2), np.float64)}
        self.h2d = self.h_poses.nbytes + self.h_opp.nbytes + self.h_nopp.nbytes
        self.d2h = sum(v.nbytes for v in self.h_out.values())

    def step(self):
        return self.planner.plan_batch(self.h_poses, self.h_opp, self.h_nopp, out=self.h_out, want_flags=True)

    def step_no_traj(self):
        """the same call without the [S,M,4] best trajectories (91 % of the result bytes)"""
        return self.planner.plan_batch(self.h_poses, self.h_opp, self.h_nopp, out=self.h_out, want_flags=True,
                                       want_traj=False)


def timed(torch, dist, dev, world_size, step, n_steps, wall=False):
    """barrier + synchronize, n_steps of step(), synchronize + barrier; max over ranks (ms).
    wall=False: CUDA events on torch's current stream (device-resident arm, launched there);
    wall=True: host clock around calls that synchronise themselves (host-buffer API)."""
    torch.cuda.synchronize(dev)
    if world_size > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if wall:
        t0 = time.perf_counter()
        for _ in range(n_steps):
            step()
        torch.cuda.synchronize(dev)
        ms = 1e3 * (time.perf_counter() - t0)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_steps):
            step()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world_size > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from f1tenth_planning_b200 import LatticePlanner, sharding
    from f1tenth_planning_b200.engine import Engine, pinned_empty

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback "
                           "(use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: run on the CPUs of the GPU's NUMA node before any pinned buffer exists
    # (first touch places the result buffers there; 8 ranks otherwise share one socket's memory)
    numa_node = sharding.bind_host_numa(local) if world_size > 1 else None
    if world_size > 1:
        # NCCL prints its version banner on stdout at VERSION level; keep stdout to the JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        # ... and whatever NCCL still writes to fd 1 while the communicator comes up goes to stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    S = args.scenarios
    track, grid, la, wd, poses, opp, n_opp = workload(rank, S)
    eng = Engine(device=local, prune_window=args.prune, **PLAN_CFG)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    C, M = eng.n_candidates, eng.n_samples

    # one nvidia-smi process on rank 0 watches every GPU of the job (eight concurrent ones on an
    # 8-GPU box took longer to start than the whole run and returned no rows)
    sampler = ClockSampler(",".join(str(i) for i in range(world_size)) if world_size > 1 else local)
    if rank == 0:
        sampler.start()

    # ---- device-resident arm -------------------------------------------------------------------
    arm = DeviceArm(torch, dev, eng, poses, opp, n_opp)
    step = arm.step
    n_warm, t_warm = 0, time.time()
    # warm-up goes on (GPU under load) until the sampler has delivered its first row, 10 s at most
    while n_warm < max(args.warmup, 3) or (rank == 0 and sampler.proc is not None and not sampler.rows
                                           and time.time() - t_warm < 10.0):
        step()
        n_warm += 1
        if n_warm % 4 == 0:
            torch.cuda.synchronize(dev)
    torch.cuda.synchronize(dev)
    # roofline denominators, measured with the GPU warm and the clock sampler running: the FFMA /
    # MUFU microbenchmarks of the library (f1l_measure_peaks); clocks of exactly this interval
    sampler.mark()
    t_pk = time.time()
    fp32_peak, mufu_peak = eng.measure_peaks()
    while time.time() - t_pk < 0.25:      # a few 50 ms sampler rows under the microbenchmark's load
        fp32_peak = max(fp32_peak, eng.measure_peaks()[0])
    peak_clocks = sampler.window() if rank == 0 else None
    step()
    torch.cuda.synchronize(dev)
    eng.set_timing(True)
    sampler.mark()
    l0 = eng.launch_count
    ms_total = timed(torch, dist, dev, world_size, step, args.steps)
    launches = eng.launch_count - l0
    clocks = sampler.window() if rank == 0 else None
    if rank == 0:
        sampler.stop()   # nvidia-smi polling the GPUs would only disturb the latency arms below
    k_sample, k_eval, k_select, n_timed = eng.mean_kernel_ms()
    eval_shape = eng.last_eval_shape()   # the template instance the timed steps launched
    eng.set_timing(False)
    value = world_size * S * C * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, arm, args.dump_outputs)   # before any later step overwrites them

    if args.quick:
        if rank == 0:
            print(json.dumps({"quick": True, "value": value, "ms_per_step": ms_total / args.steps,
                              "kernels_ms": {"sample": k_sample, "eval": k_eval, "select": k_select},
                              "kernel": eval_shape["name"], "fp32_peak": fp32_peak, "clocks": clocks,
                              "checksum": float(arm.o_costs[torch.isfinite(arm.o_costs)].double().sum().item()),
                              "best_idx_sum": int(arm.o_idx.long().sum().item())}), flush=True)
        if world_size > 1:
            dist.destroy_process_group()
        return
    flags = arm.o_flags.cpu().numpy()
    # work counters of the deviation pass from one extra, untimed step (counting is off in the
    # timed ones: it costs every CTA a barrier and two global atomics)
    eng.set_stats(True)
    step()
    torch.cuda.synchronize(dev)
    seg_steps, seg_cands = eng.stats()
    eng.set_stats(False)
    # window segments each valid candidate was tested against (= W unless --prune 1)
    w_eff = seg_steps / seg_cands if seg_cands else float(PLAN_CFG["window"])
    step_flops, valid_frac, mean_passes = work_flops(flags, M, seg_steps, float(n_opp.mean()))
    achieved_tflops = step_flops / (k_eval * 1e-3) / 1e12 if k_eval > 0 else None
    # the same without the work the kernel mostly skips: the 16 P M grid-probe FLOPs (a clearance
    # lookup proves most footprints free) and the 6 K M opponent broad-phase FLOPs (candidate-level
    # prune) -- the conservative reading of the roofline fraction
    n_full = int(((flags & 1) != 0).sum())
    skippable = n_full * M * (16.0 * F.P_PROBES + 6.0 * float(n_opp.mean()))
    achieved_noskip = (step_flops - skippable) / (k_eval * 1e-3) / 1e12 if k_eval > 0 else None
    mufu_ops = float((flags >> 4).astype(np.float64).sum()) * (2 * F.Q_NEWTON + 1) + flags.size * 5.0 * M

    # ---- side measurement: the same step with prune_window = 1 (bit-identical costs) ------------
    pruned = None
    if world_size == 1 and not args.no_extras and not args.prune:
        costs_full = arm.o_costs.clone()
        eng.configure(prune_window=1)
        for _ in range(3):
            step()
        torch.cuda.synchronize(dev)
        eng.set_timing(True)
        p_ms = timed(torch, dist, dev, 1, step, args.steps) / args.steps
        _, pk_eval, _, _ = eng.mean_kernel_ms()
        eng.set_timing(False)
        eng.set_stats(True)
        step()
        torch.cuda.synchronize(dev)
        ps, pc = eng.stats()
        eng.set_stats(False)
        p_flops, _, _ = work_flops(flags, M, ps, float(n_opp.mean()))
        pruned = {"candidates_per_s": S * C / (p_ms * 1e-3), "ms_per_step": p_ms, "eval_kernel_ms": pk_eval,
                  "window_segments_tested_mean": ps / max(pc, 1),
                  "candidates_in_deviation_pass": int(pc),
                  "valid_candidates": int(((flags & 1) != 0).sum()),
                  "executed_tflops": p_flops / (pk_eval * 1e-3) / 1e12,
                  "costs_bit_identical_to_full_scan": bool(torch.equal(arm.o_costs, costs_full))}
        eng.configure(prune_window=0)
        step()
        torch.cuda.synchronize(dev)
    hbm_bytes = S * C * F.candidate_hbm_bytes() + S * (M * 16 + 32 + 4 + 4 + 16) + S * (32 + K_OPP * 24 + 4)

    # ---- end-to-end arm: public API, pinned host buffers, H2D + D2H inside the timed region ------
    planner = LatticePlanner(waypoints=track, device=local, **PLAN_CFG)
    planner.set_map(*grid)
    planner.set_goal_grid(la, wd)
    host = HostArm(planner, pinned_empty, poses, opp, n_opp)
    for _ in range(2):
        host.step()
    e2e_steps = max(3, min(args.steps, 10))
    t_e2e = timed(torch, dist, dev, world_size, host.step, e2e_steps, wall=True) * 1e-3
    e2e_value = world_size * S * C * e2e_steps / t_e2e
    assert np.array_equal(host.h_out["best_idx"], arm.o_idx.cpu().numpy()), "e2e and device-resident arms disagree"
    assert np.array_equal(host.h_out["flags"], flags), "e2e and device-resident arms disagree (flags)"
    # side measurement: the same call with want_traj=False -- what the end-to-end rate is when the
    # host link does not have to carry the best trajectories (it is the bound at N = 8 on this box)
    host.step_no_traj()
    t_nt = timed(torch, dist, dev, world_size, host.step_no_traj, e2e_steps, wall=True) * 1e-3
    e2e_no_traj = {"value": world_size * S * C * e2e_steps / t_nt, "unit": UNIT,
                   "d2h_bytes_per_step": host.d2h - host.h_out["best_traj"].nbytes}

    # ---- what the host link gives: every rank copies 128 MB device -> pinned host at the same time
    #      (the e2e arm's result copy is 176 MB per step per GPU) ----------------------------------
    probe_dev = torch.empty(128 << 20, dtype=torch.uint8, device=dev)
    probe_host = torch.empty(128 << 20, dtype=torch.uint8, pin_memory=True)
    probe_host.copy_(probe_dev)
    probe_ms = timed(torch, dist, dev, world_size, lambda: probe_host.copy_(probe_dev, non_blocking=True), 4)
    d2h_probe_gbs = 4 * (128 << 20) / (probe_ms * 1e-3) / 1e9
    del probe_dev, probe_host

    # ---- strong scaling (BASELINE config 4 as written): the 10^5 scenarios of rank 0's set split
    #      into contiguous blocks over the ranks, same two arms --------------------------------------
    strong = None
    if world_size > 1:
        _, _, _, _, poses0, opp0, n_opp0 = workload(0, S)
        lo, hi = sharding.block(S, rank, world_size)
        sarm = DeviceArm(torch, dev, eng, poses0[lo:hi].copy(), opp0[lo:hi].copy(), n_opp0[lo:hi].copy())
        for _ in range(3):
            sarm.step()
        s_ms = timed(torch, dist, dev, world_size, sarm.step, args.steps) / args.steps
        shost = HostArm(planner, pinned_empty, poses0[lo:hi], opp0[lo:hi], n_opp0[lo:hi])
        for _ in range(2):
            shost.step()
        s_e2e = timed(torch, dist, dev, world_size, shost.step, e2e_steps, wall=True) * 1e-3 / e2e_steps
        one_gpu_ms = ms_total / args.steps          # 10^5 scenarios on ONE GPU: this run's weak step
        strong = {"scaling": "strong", "scenarios_total": S, "scenarios_per_rank": hi - lo,
                  "value": S * C / (s_ms * 1e-3), "unit": UNIT, "ms_per_step": s_ms,
                  "one_gpu_ms_per_step_same_run": one_gpu_ms,
                  "efficiency_vs_one_gpu_same_run": one_gpu_ms / (world_size * s_ms),
                  "e2e": {"value": S * C / s_e2e, "unit": UNIT, "h2d_bytes_per_step": shost.h2d,
                          "d2h_bytes_per_step": shost.d2h,
                          "efficiency_vs_one_gpu_same_run": (t_e2e / e2e_steps) / (world_size * s_e2e)}}
        del sarm, shost

    sharded = None
    if world_size > 1 and not args.no_extras:
        try:
            sharded = sharded_dense_query(track, grid, local, rank, world_size, dev)
        except Exception as e:   # the headline line must not depend on the side measurement
            sharded = {"c5_sharded_error": "%s: %s" % (type(e).__name__, e)}

    if rank != 0:
        if world_size > 1:
            dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps,
        "warmup": max(args.warmup, 3), "warmup_steps_run": n_warm, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": "c4: %d independent scenarios per GPU x 4x7 goal grid (%d candidates/step/GPU), "
                        "M=%d arc samples, raceline window W=%d (prune_window=%d: %.1f segments tested per "
                        "sample), 1..%d opponents, occupancy grid on, "
                        "kappa_max off (every converged candidate does the full cost+collision work)"
                        % (S, S * C, M, PLAN_CFG["window"], args.prune, w_eff, K_OPP),
            "track": "ellipse N=2000 a=80 b=40", "grid": "3400x1800 @0.05 m",
            "valid_frac": valid_frac, "newton_passes_mean": mean_passes,
            "feasible_frac": float(np.isfinite(arm.o_costs.cpu().numpy()).mean()),
            "l2": "per-step working set %.0f MB > 126 MB L2 (outputs rewritten every step); no explicit flush"
                  % ((hbm_bytes + S * C * 4) / 1e6),
            "host_numa_node": numa_node,
        },
        "roofline": {
            "bound": "fp32", "achieved": achieved_tflops, "peak": fp32_peak, "unit": "TFLOP/s",
            "frac": achieved_tflops / fp32_peak if achieved_tflops else None,
            "peak_source": "FFMA microbenchmark measured in this run with the GPU warm "
                           "(f1l_measure_peaks, best of the launches in a 0.25 s window); "
                           "MEASURED_PEAKS.json has no FP32 entry; nominal 74.4",
            "peak_clocks": peak_clocks,
            # conservative reading: grid-probe and opponent broad-phase FLOPs of the model left out
            # (the clearance map / candidate-level prune skip nearly all of them)
            "achieved_without_skippable_flops": achieved_noskip,
            "frac_without_skippable_flops": achieved_noskip / fp32_peak if achieved_noskip else None,
            "kernel": eval_shape["name"], "kernel_plan": eval_shape, "kernel_ms": k_eval, "kernel_launches_timed": n_timed,
            "kernel_share_of_step": k_eval / (ms_total / args.steps) if k_eval else None,
            "flops_per_launch": step_flops,
            # the secondary roofline SURVEY 8d names: MUFU (sin / cos / sqrt) operations of the
            # step -- (2 Q + 1) per Newton pass and 5 per arc sample -- against the measured pipe peak
            "mufu": {"achieved_gops": mufu_ops / (k_eval * 1e-3) / 1e9 if k_eval > 0 else None,
                     "peak_gops": mufu_peak,
                     "frac": mufu_ops / (k_eval * 1e-3) / 1e9 / mufu_peak if (k_eval > 0 and mufu_peak) else None},
            "mufu_peak_gops": mufu_peak,
            # dram__bytes_read.sum + dram__bytes_write.sum of one eval_kernel launch of this workload
            # (ncu --set full; profiles/) -- bench.py cannot run under ncu itself
            "traffic": profiled_dram_bytes() if (S == S_PER_GPU and not args.prune) else None,
            "traffic_source": PROFILE_MD,
            "hbm": {"algorithmic_bytes_per_step": hbm_bytes,
                    "achieved_gbs": hbm_bytes / (ms_total / args.steps * 1e-3) / 1e9},
        },
        "kernels_ms": {"sample": k_sample, "eval": k_eval, "select": k_select},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": host.h2d,
                "d2h_bytes_per_step": host.d2h, "steps": e2e_steps,
                "d2h_gbs_per_gpu": host.d2h / (t_e2e / e2e_steps) / 1e9,
                # plain 128 MB device -> pinned-host copies issued by all ranks at the same time
                "d2h_link_probe_gbs_per_gpu": d2h_probe_gbs,
                # side measurement, not the headline: want_traj=False
                "without_best_traj": e2e_no_traj,
                "api": "LatticePlanner.plan_batch (pinned host buffers; every output of the "
                       "device-resident arm, flags included)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if strong is not None:
        line["strong"] = strong
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            mp = json.load(f)
        line["roofline"]["hbm"]["peak_gbs"] = mp.get("hbm_gbs")
        line["roofline"]["hbm"]["frac"] = line["roofline"]["hbm"]["achieved_gbs"] / mp["hbm_gbs"]
    except Exception:
        line["roofline"]["hbm"]["peak_gbs"] = 6650.0
        line["roofline"]["hbm"]["note"] = "fallback peak"
    if world_size == 1 and not args.no_cpu_baseline:
        v, n, th, dt = cpu_reference_rate(track, grid, la, wd, poses, opp, n_opp, seconds=12.0)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": th, "kind": "port",
                                "sample": "the first %d of the %d scenarios (x%d candidates), %.1f s, C oracle "
                                          "(oracle/c/f1o.c) with OpenMP over scenarios" % (n, S, C, dt)}
    if sharded is not None:
        line["extra"] = sharded
    if world_size == 1 and not args.no_extras:
        try:
            line["extra"] = extras(track, grid, local, fp32_peak)
        except Exception as ex:  # side measurements must not lose the headline
            line["extra"] = {"error": repr(ex)}
        if pruned is not None:
            line["extra"]["prune_window_1"] = pruned
    print(json.dumps(line), flush=True)
    if world_size > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: self-launch one rank per GPU the way the driver does
        port = str(29500 + (os.getpid() % 2000))
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
                                   "--master-port", port, os.path.abspath(__file__)] + sys.argv[1:])
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
