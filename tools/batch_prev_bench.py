"""Cost of per-scenario previous paths in batch planning, measured at bench.py's workload.

The same engine and scenarios as bench.py (10^5 scenarios x 28 candidates, M = 100, W = 128, up
to 8 opponents, corridor grid, synth.scenario_batch seeds), four arms alternated in one process:
    dev        plan_batch_dev, no previous path (bench.py's device-resident step)
    dev_prev   plan_batch_dev with a [S,M] f32 path and [S] u8 flag per scenario, update_prev=1
    host       LatticePlanner.plan_batch with pinned host buffers, no previous path
    host_prev  the same with pinned [S,M] / [S] previous paths, update_prev=True
Each round runs every arm for --steps steps after its own warm-up; device arms are timed with
CUDA events (and the library's per-kernel events), host arms with a host clock around calls that
synchronise.  The per-scenario paths add 400 B read + 400 B written per scenario to the device
step, and 2 x 400 B per scenario over the host link to the host step.  Prints one JSON line
(and writes it to --out): per-arm mean and per-round step times, the overheads, the card name
and its power limit.  Needs a CUDA device; there is no CPU fallback.

    python tools/batch_prev_bench.py --steps 10 --rounds 3 --out batch_prev.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload, engine config and arms of the headline benchmark)


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=bench.S_PER_GPU)
    ap.add_argument("--steps", type=int, default=10, help="timed steps per arm per round")
    ap.add_argument("--warmup", type=int, default=2, help="untimed steps before each timed arm")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the four arms")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.rounds < 1:
        ap.error("--steps and --rounds must be >= 1")

    import torch
    from f1tenth_planning_b200 import LatticePlanner
    from f1tenth_planning_b200.engine import Engine, pinned_empty
    if not torch.cuda.is_available():
        raise RuntimeError("batch_prev_bench.py needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    S = args.scenarios
    track, grid, la, wd, poses, opp, n_opp = bench.workload(0, S)
    eng = Engine(device=local, **bench.PLAN_CFG)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    M = eng.n_samples

    arm = bench.DeviceArm(torch, dev, eng, poses, opp, n_opp)
    d_prev = torch.zeros(S, M, dtype=torch.float32, device=dev)
    d_valid = torch.zeros(S, dtype=torch.uint8, device=dev)

    def dev_prev():
        eng.plan_batch_dev(arm.tp, arm.to, arm.tn, best_idx=arm.o_idx, best_cost=arm.o_cost,
                           best_traj=arm.o_traj, costs=arm.o_costs, flags=arm.o_flags,
                           steer_speed=arm.o_ss, prev_theta=d_prev, has_prev=d_valid, update_prev=True)

    planner = LatticePlanner(waypoints=track, device=local, **bench.PLAN_CFG)
    planner.set_map(*grid)
    planner.set_goal_grid(la, wd)
    host = bench.HostArm(planner, pinned_empty, poses, opp, n_opp)
    h_prev = pinned_empty((S, M), np.float32)
    h_prev[:] = 0.0
    h_valid = pinned_empty((S,), np.uint8)
    h_valid[:] = 0

    def host_prev():
        planner.plan_batch(host.h_poses, host.h_opp, host.h_nopp, out=host.h_out, want_flags=True,
                           prev_theta=h_prev, has_prev=h_valid, update_prev=True)

    arms = {"dev": (arm.step, False), "dev_prev": (dev_prev, False),
            "host": (host.step, True), "host_prev": (host_prev, True)}
    ms = {k: [] for k in arms}
    eval_ms = {"dev": [], "dev_prev": []}
    for _ in range(args.rounds):
        for name, (step, wall) in arms.items():
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize(dev)
            if not wall:
                eng.set_timing(True)
            ms[name].append(bench.timed(torch, None, dev, 1, step, args.steps, wall=wall) / args.steps)
            if not wall:
                eval_ms[name].append(eng.mean_kernel_ms()[1])
                eng.set_timing(False)
    assert bool(d_valid.all()) and bool(h_valid.all())

    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    spread = {k: float(np.max(v) - np.min(v)) for k, v in ms.items()}
    line = {
        "workload": "bench.py c4: %d scenarios x %d candidates, M=%d, W=%d, <=%d opponents, corridor grid"
                    % (S, eng.n_candidates, M, bench.PLAN_CFG["window"], bench.K_OPP),
        "steps_per_arm_per_round": args.steps, "rounds": args.rounds,
        "ms_per_step_mean": mean, "ms_per_step_rounds": ms, "ms_per_step_spread": spread,
        "eval_kernel_ms_mean": {k: float(np.mean(v)) for k, v in eval_ms.items()},
        "overhead_dev": mean["dev_prev"] / mean["dev"] - 1.0,
        "overhead_host": mean["host_prev"] / mean["host"] - 1.0,
        "extra_bytes_per_step": {"hbm": 2 * S * (4 * M + 1), "host_link": 2 * S * (4 * M + 1)},
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
