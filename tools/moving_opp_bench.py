"""What constant-velocity opponent prediction costs, measured at bench.py's workload, and what it
changes in closed-loop races.

Batch arms (10^5 scenarios x 28 candidates, M = 100, W = 128, up to 8 opponents, corridor grid,
bench.py's scenarios), alternated in one process:
    static   plan_batch_dev (bench.py's device-resident step)
    moving   plan_batch_dev with every opponent moving at U(2, 8) m/s along its heading
             (synth.opponent_velocities), v_min = 1 m/s
Each round runs both arms after their own warm-up; step times come from CUDA events.  A separate
torch.profiler pass (no step timing) reports the mean eval_kernel time per arm.

Fleet arms: --fleet-cars cars in races of 4 on the same track, --fleet-steps planning steps, with
predict off and on: ms per step, cars frozen by a car-to-car collision, mean progress.

Prints one JSON line (and writes it to --out) with the card's name and power limit read in the same
run.  Needs a CUDA device; there is no CPU fallback.

    python tools/moving_opp_bench.py --steps 10 --rounds 3 --out moving_opp.json
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload and engine config of the headline benchmark)
from tools.batch_prev_bench import card  # noqa: E402
from tools.rollout_bench import event_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=bench.S_PER_GPU)
    ap.add_argument("--steps", type=int, default=10, help="timed steps per batch arm per round")
    ap.add_argument("--warmup", type=int, default=2, help="untimed steps before each timed arm")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the batch arms")
    ap.add_argument("--fleet-cars", type=int, default=10000)
    ap.add_argument("--fleet-steps", type=int, default=200)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.rounds < 1 or args.fleet_steps < 1 or args.fleet_cars % 4:
        ap.error("--steps, --rounds, --fleet-steps must be >= 1 and --fleet-cars a multiple of 4")

    import torch
    from torch.profiler import ProfilerActivity, profile
    from f1tenth_planning_b200 import synth
    from f1tenth_planning_b200.engine import Engine
    from f1tenth_planning_b200.rollout import CAR_HIT_CAR
    if not torch.cuda.is_available():
        raise RuntimeError("moving_opp_bench.py needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    S = args.scenarios
    track, grid, la, wd, poses, opp, n_opp = bench.workload(0, S)
    eng = Engine(device=local, **bench.PLAN_CFG)
    eng.set_track(track)
    eng.set_grid(*grid)
    eng.set_goal_grid(la, wd)
    C = eng.n_candidates
    arm = bench.DeviceArm(torch, dev, eng, poses, opp, n_opp)
    vel = torch.from_numpy(synth.opponent_velocities(track, opp, np.random.default_rng(21), 2.0, 8.0)).to(dev)

    def batch_step(v):
        def step():
            eng.plan_batch_dev(arm.tp, arm.to, arm.tn, best_idx=arm.o_idx, best_cost=arm.o_cost,
                               best_traj=arm.o_traj, costs=arm.o_costs, flags=arm.o_flags,
                               steer_speed=arm.o_ss, opponent_velocities=v)
        return step

    arms = {"static": batch_step(None), "moving": batch_step(vel)}
    ms = {k: [] for k in arms}
    collide = {}
    for _ in range(args.rounds):
        for name, step in arms.items():
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize(dev)
            ms[name].append(bench.timed(torch, None, dev, 1, step, args.steps, wall=False) / args.steps)
            f = arm.o_flags.cpu().numpy()
            valid = (f & 1) != 0
            collide[name] = float(((f & 2) != 0)[valid].mean())

    # eval_kernel alone, torch.profiler in a pass of its own
    eval_us = {}
    for name, step in arms.items():
        step()
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                step()
            torch.cuda.synchronize(dev)
        ev = [e for e in prof.events() if e.device_type.name == "CUDA" and "eval_kernel" in e.name]
        eval_us[name] = float(np.mean([e.device_time for e in ev])) if ev else None

    # fleets: races of 4, predict off and on
    rng = np.random.default_rng(5)
    n = track.shape[0]
    G = 4
    base = np.repeat(rng.integers(0, n, args.fleet_cars // G), G)
    idx = (base + 12 * np.tile(np.arange(G), args.fleet_cars // G)) % n
    psi = track[idx, 3]
    off = rng.normal(0.0, 0.25, args.fleet_cars)
    X0 = np.stack([track[idx, 0] - off * np.sin(psi), track[idx, 1] + off * np.cos(psi), psi,
                   np.full(args.fleet_cars, 5.0)], axis=1)
    fleet = {}
    for name, predict in (("predict_off", False), ("predict_on", True)):
        f = eng.fleet(X0, group=G)
        f.run(1, predict=predict)   # warm-up: buffers, modules
        f = eng.fleet(X0, group=G)
        torch.cuda.synchronize(dev)
        t = event_ms(torch, lambda: f.run(args.fleet_steps, predict=predict))
        st = f.status.cpu().numpy()
        fleet[name] = {"ms_per_step": t / args.fleet_steps,
                       "cars_hit_car": int(((st & CAR_HIT_CAR) != 0).sum()),
                       "mean_progress_m": float(f.progress.cpu().numpy().mean())}

    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    line = {
        "workload": "bench.py c4: %d scenarios x %d candidates, M=%d, W=%d, <=%d opponents, corridor grid; "
                    "moving: U(2, 8) m/s along the heading, v_min = 1" % (S, C, eng.n_samples,
                                                                         bench.PLAN_CFG["window"], bench.K_OPP),
        "steps_per_arm_per_round": args.steps, "rounds": args.rounds,
        "ms_per_step_mean": mean, "ms_per_step_rounds": ms,
        "ms_per_step_spread": {k: float(np.max(v) - np.min(v)) for k, v in ms.items()},
        "overhead_moving": mean["moving"] / mean["static"] - 1.0,
        "eval_kernel_us_profiler": eval_us,
        "opp_collision_share_of_valid_last_step": collide,
        "fleet": dict(cars=args.fleet_cars, group=G, steps=args.fleet_steps, **fleet),
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
