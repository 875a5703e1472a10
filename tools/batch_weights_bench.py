"""Cost of per-scenario cost weights and per-term costs in batch planning, measured at bench.py's
workload.

The same engine and scenarios as bench.py (10^5 scenarios x 28 candidates, M = 100, W = 128, up
to 8 opponents, corridor grid, synth.scenario_batch seeds), arms alternated in one process:
    dev             plan_batch_dev, no weights (bench.py's device-resident step)
    dev_w_config    the same with the config's weights broadcast to a [S,5] f32 tensor
    dev_w_random    the same with random per-scenario weights
    dev_terms, dev_w_config_terms, dev_w_random_terms
                    the three above with the [S,C,5] f32 per-term costs requested
    fleet, fleet_w  Fleet.run of 10^5 cars in races of 4 (tools/rollout_bench.py arm (a)) without
                    and with random per-car weights, --fleet-steps planning steps per timed call
Each round runs every arm after its own warm-up; device times per step come from CUDA events, the
eval kernel's from the library's per-kernel events.  Weights add one 20-byte load per eval CTA;
terms add S x C x 20 bytes of writes per step.  Prints one JSON line (and writes it to --out) with
the card's name and power limit read in the same run.  Needs a CUDA device; there is no CPU fallback.

    python tools/batch_weights_bench.py --steps 10 --rounds 3 --out batch_weights.json
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload, engine config and arms of the headline benchmark)
from tools.batch_prev_bench import card  # noqa: E402
from tools.rollout_bench import event_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=bench.S_PER_GPU)
    ap.add_argument("--steps", type=int, default=10, help="timed steps per batch arm per round")
    ap.add_argument("--warmup", type=int, default=2, help="untimed steps before each timed arm")
    ap.add_argument("--fleet-steps", type=int, default=20, help="planning steps per timed Fleet.run")
    ap.add_argument("--group", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the arms")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.rounds < 1 or args.fleet_steps < 1:
        ap.error("--steps, --fleet-steps and --rounds must be >= 1")

    import torch
    from f1tenth_planning_b200.engine import Engine
    if not torch.cuda.is_available():
        raise RuntimeError("batch_weights_bench.py needs a CUDA device")
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
    w_cfg = torch.tensor(list(eng.config.weights), dtype=torch.float32, device=dev).expand(S, 5).contiguous()
    rng = np.random.default_rng(11)
    w_rnd = torch.from_numpy(rng.uniform(0.0, 2.0, (S, 5)).astype(np.float32)).to(dev)
    terms = torch.empty(S, C, 5, dtype=torch.float32, device=dev)

    def batch_step(weights, want_terms):
        def step():
            eng.plan_batch_dev(arm.tp, arm.to, arm.tn, best_idx=arm.o_idx, best_cost=arm.o_cost,
                               best_traj=arm.o_traj, costs=arm.o_costs, flags=arm.o_flags,
                               steer_speed=arm.o_ss, weights=weights,
                               terms=terms if want_terms else None)
        return step

    batch_arms = {"dev": batch_step(None, False), "dev_w_config": batch_step(w_cfg, False),
                  "dev_w_random": batch_step(w_rnd, False), "dev_terms": batch_step(None, True),
                  "dev_w_config_terms": batch_step(w_cfg, True),
                  "dev_w_random_terms": batch_step(w_rnd, True)}

    # rollout arm (a) of tools/rollout_bench.py: 10^5 cars in races of --group
    fleets = {"fleet": eng.fleet(poses, group=args.group),
              "fleet_w": eng.fleet(poses, group=args.group, weights=w_rnd)}
    for f in fleets.values():
        f.run(2)   # warm-up: buffers, modules

    ms = {k: [] for k in list(batch_arms) + list(fleets)}
    eval_ms = {k: [] for k in batch_arms}
    for _ in range(args.rounds):
        for name, step in batch_arms.items():
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize(dev)
            eng.set_timing(True)
            ms[name].append(bench.timed(torch, None, dev, 1, step, args.steps, wall=False) / args.steps)
            eval_ms[name].append(eng.mean_kernel_ms()[1])
            eng.set_timing(False)
        for name, f in fleets.items():
            torch.cuda.synchronize(dev)
            ms[name].append(event_ms(torch, lambda: f.run(args.fleet_steps)) / args.fleet_steps)
    for f in fleets.values():
        assert bool(torch.isfinite(f.state).all())

    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    spread = {k: float(np.max(v) - np.min(v)) for k, v in ms.items()}
    line = {
        "workload": "bench.py c4: %d scenarios x %d candidates, M=%d, W=%d, <=%d opponents, corridor grid"
                    % (S, C, eng.n_samples, bench.PLAN_CFG["window"], bench.K_OPP),
        "fleet": "%d cars in races of %d, %d steps per timed call" % (S, args.group, args.fleet_steps),
        "steps_per_arm_per_round": args.steps, "rounds": args.rounds,
        "ms_per_step_mean": mean, "ms_per_step_rounds": ms, "ms_per_step_spread": spread,
        "eval_kernel_ms_mean": {k: float(np.mean(v)) for k, v in eval_ms.items()},
        "overhead": {k: mean[k] / mean["dev"] - 1.0 for k in batch_arms if k != "dev"},
        "overhead_fleet_w": mean["fleet_w"] / mean["fleet"] - 1.0,
        "extra_bytes_per_step": {"weights": S * 20, "terms": S * C * 20},
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
