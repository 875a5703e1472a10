"""Closed-loop rollouts on the device (Fleet.run, f1l_rollout_dev): what the step kernel and the
device-resident loop cost.

(a) throughput: 10^5 cars in races of 4 on bench.py's ellipse, corridor grid, goal grid and planner
    configuration (the cars start at bench.py's seeded scenario poses), --steps planning steps.
    Device time per step (CUDA events) of Fleet.run against f1l_plan_batch_prev_dev alone on the
    same fleet state (the races' opponents uploaded once, previous paths updated in place), and the
    mean device time of rollout_step_kernel from a torch.profiler pass of its own.  With
    --vehicle st a fleet of dynamic single-track cars (rollout.Vehicle's defaults) at the same poses
    is timed as a third arm, alternated with the others, and each model's rollout_step_kernel
    instance gets a profiler pass of its own.
(b) latency: 32 cars, --long-steps steps, wall time per step (host clock around calls that end in a
    device synchronise) of one Fleet.run call against the Python loop of the batch planner's
    device-resident test: plan_batch_dev + a kinematic bicycle in torch, one step at a time.
Arms alternate for --rounds rounds.  Prints one JSON line (and writes it to --out) with the card's
name and power limit read in the same run.  Needs a CUDA device; there is no CPU fallback.

    python tools/rollout_bench.py --out rollout.json
    python tools/rollout_bench.py --vehicle st --out rollout_st.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload and engine config of the headline benchmark)
from tools.batch_prev_bench import card  # noqa: E402

DT, WHEELBASE = 0.01, 0.33


def race_opponents(torch, dev, poses, G):
    """[S,16,3] f64 / [S] i32: the other cars of each car's race in race order"""
    S = poses.shape[0]
    R = poses[:, :3].reshape(S // G, G, 3)
    opp = np.zeros((S, 16, 3))
    for j in range(G):
        opp[j::G, :G - 1] = np.delete(R, j, axis=1)
    return (torch.from_numpy(opp).to(dev),
            torch.full((S,), G - 1, dtype=torch.int32, device=dev))


def event_ms(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def wall_ms(torch, dev, fn):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize(dev)
    return 1e3 * (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cars", type=int, default=100000)
    ap.add_argument("--group", type=int, default=4)
    ap.add_argument("--steps", type=int, default=20, help="(a) planning steps per timed call")
    ap.add_argument("--long-cars", type=int, default=32)
    ap.add_argument("--long-steps", type=int, default=500, help="(b) planning steps per timed call")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--vehicle", choices=("kinematic", "st"), default="kinematic",
                    help="st: also time (a) with the dynamic single-track model")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    from f1tenth_planning_b200.engine import Engine
    from f1tenth_planning_b200.rollout import Vehicle
    if not torch.cuda.is_available():
        raise RuntimeError("rollout_bench.py needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    track, grid, la, wd, poses, _, _ = bench.workload(0, args.cars)
    eng = Engine(device=local, **bench.PLAN_CFG)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    S, G, T, M = args.cars, args.group, args.steps, eng.n_samples

    # (a) the fleet's own steps against the planner alone on the same state
    fleet = eng.fleet(poses, group=G)
    fleet.run(2)   # warm-up: buffers, modules
    fleets = {"fleet_run": fleet}
    if args.vehicle == "st":
        fleets["fleet_run_st"] = eng.fleet(poses, group=G, vehicle=Vehicle())
        fleets["fleet_run_st"].run(2)
    opp, n_opp = race_opponents(torch, dev, fleet.state.cpu().numpy(), G)
    P = fleet.prev_theta.clone()
    V = fleet.has_prev.clone()
    o_idx = torch.empty(S, dtype=torch.int32, device=dev)
    o_cost = torch.empty(S, dtype=torch.float32, device=dev)
    o_ss = torch.empty(S, 2, dtype=torch.float64, device=dev)

    def plan_only():
        for _ in range(T):
            eng.plan_batch_dev(fleet.state, opp, n_opp, best_idx=o_idx, best_cost=o_cost,
                               steer_speed=o_ss, prev_theta=P, has_prev=V, update_prev=True)

    plan_only()
    ms_a = {name: [] for name in fleets}
    ms_a["plan_batch_prev_dev"] = []
    for _ in range(args.rounds):
        for name, f in fleets.items():
            ms_a[name].append(event_ms(torch, lambda: f.run(T)) / T)
        ms_a["plan_batch_prev_dev"].append(event_ms(torch, plan_only) / T)
    for f in fleets.values():
        assert torch.isfinite(f.state).all() and (f.dyn is None or torch.isfinite(f.dyn).all())
    from torch.profiler import profile, ProfilerActivity
    step_us = {}
    for name, f in fleets.items():   # one pass per model: the instances' names differ by template only
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            f.run(T)
            torch.cuda.synchronize(dev)
        us = [e.device_time_total / e.count for e in prof.key_averages() if "rollout_step_kernel" in e.key]
        step_us[name] = us[0] if us else None

    # (b) one Fleet.run call against the Python loop with a torch bicycle
    Sb, Tb = args.long_cars, args.long_steps
    lp = poses[:Sb]
    fb = eng.fleet(lp, group=1)
    fb.run(2)
    tX = torch.from_numpy(lp).to(dev)
    tP = torch.zeros(Sb, M, dtype=torch.float32, device=dev)
    tV = torch.zeros(Sb, dtype=torch.uint8, device=dev)
    b_idx = torch.empty(Sb, dtype=torch.int32, device=dev)
    b_cost = torch.empty(Sb, dtype=torch.float32, device=dev)
    b_ss = torch.empty(Sb, 2, dtype=torch.float64, device=dev)

    def torch_loop():
        X = tX
        for _ in range(Tb):
            eng.plan_batch_dev(X, best_idx=b_idx, best_cost=b_cost, steer_speed=b_ss, prev_theta=tP,
                               has_prev=tV, update_prev=True)
            steer = b_ss[:, 0].clamp(-0.4189, 0.4189)
            v = X[:, 3] + (b_ss[:, 1] - X[:, 3]).clamp(-9.51 * DT, 9.51 * DT)
            X = torch.stack([X[:, 0] + v * torch.cos(X[:, 2]) * DT, X[:, 1] + v * torch.sin(X[:, 2]) * DT,
                             X[:, 2] + v / WHEELBASE * torch.tan(steer) * DT, v], dim=1)

    torch_loop()
    ms_b = {"fleet_run": [], "torch_loop": []}
    for _ in range(args.rounds):
        ms_b["fleet_run"].append(wall_ms(torch, dev, lambda: fb.run(Tb)) / Tb)
        ms_b["torch_loop"].append(wall_ms(torch, dev, torch_loop) / Tb)

    mean = lambda d: {k: float(np.mean(v)) for k, v in d.items()}   # noqa: E731
    line = {
        "a_workload": "%d cars in races of %d, bench.py ellipse + corridor, %d candidates, M=%d, %d steps"
                      % (S, G, eng.n_candidates, M, T),
        "a_device_ms_per_step": mean(ms_a), "a_device_ms_per_step_rounds": ms_a,
        "a_step_kernel_us_profiler": step_us["fleet_run"],
        "a_step_kernel_us_profiler_st": step_us.get("fleet_run_st"),
        "b_workload": "%d cars, %d steps" % (Sb, Tb),
        "b_wall_ms_per_step": mean(ms_b), "b_wall_ms_per_step_rounds": ms_b,
        "card": card(local), "device_name": torch.cuda.get_device_name(dev),
    }
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
