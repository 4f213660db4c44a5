"""Time batched MPPI (opendog_b200.mppi.BatchedMPPI) on the GPU: one plan (broadcast + rollout + reduce) and one
closed-loop control step (plan + the robots' step + shift + reset of ended episodes), each as CUDA-graph replays timed
with CUDA events, for K robots x `--samples` samples x horizon `--horizon`.

    python tools/bench_mppi_batched.py [--robots 1 4 16 64] [--samples 1024] [--horizon 64] [--replays 20]

Prints the GPU's name and power limit, then per K: ms per plan, ms per robot-plan, robot-plans/s and ms per control step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from opendog_b200.env import BatchedWalkEnv  # noqa: E402
from opendog_b200.mppi import BatchedMPPI  # noqa: E402


def gpu_description():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def time_replays(fn, replays):
    fn(); fn(); fn()                          # eager warm-up, capture, first replay
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(replays):
        fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / replays


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, nargs="+", default=[1, 4, 16, 64])
    ap.add_argument("--samples", type=int, default=1024)
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--replays", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mppi_batched needs a CUDA device")
    name, power = gpu_description()
    print(f"GPU: {name}, power limit {power}")
    print(f"{'K':>4} {'ms/plan':>10} {'ms/robot-plan':>14} {'robot-plans/s':>14} {'ms/control step':>16}")
    for K in args.robots:
        robots = BatchedWalkEnv(K, seed=0, info_keys=None)
        robots.reset()
        for _ in range(12):                   # landed robots as the start states
            robots.step(torch.zeros(K, robots.act_dim, device=robots.device))
        plan = BatchedMPPI(robots, samples_per_robot=args.samples, horizon=args.horizon, seed=0, use_graph=True)
        ms_plan = time_replays(plan.plan, args.replays)
        ctl = BatchedMPPI(robots, samples_per_robot=args.samples, horizon=args.horizon, seed=0, use_graph=True)
        ms_ctl = time_replays(ctl.control_step, args.replays)
        row = dict(robots=K, samples_per_robot=args.samples, horizon=args.horizon, replays=args.replays,
                   ms_per_plan=round(ms_plan, 3), ms_per_robot_plan=round(ms_plan / K, 3),
                   robot_plans_per_s=round(1e3 * K / ms_plan, 1), ms_per_control_step=round(ms_ctl, 3),
                   gpu=name, power_limit=power)
        print(f"{K:>4} {ms_plan:>10.2f} {ms_plan / K:>14.3f} {1e3 * K / ms_plan:>14.1f} {ms_ctl:>16.2f}")
        print(json.dumps(row), flush=True)
        del plan, ctl, robots
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
