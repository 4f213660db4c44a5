"""Time the terrain trainer's policy forward (12-1024-512-8) and the on-device rollouts of both QuadrupedEnv trainers.

    python tools/bench_policy_wide.py [--rows 4096,16384,65536] [--envs 4096] [--horizon 24] [--out FILE.json]

Prints one JSON object:
  * forward: device-timed ms per call (CUDA events over `--iters` calls after a warm-up) of `ActorCriticB200.act` with the
    fused 1024 / 512 kernel and with `_act_library` (bf16 autocast GEMMs through torch) at each row count;
  * collect: device-timed ms per policy step of `Rollout.collect` (graph replays) for BatchedQuadrupedEnv with the
    22-512-256-4 policy and BatchedTerrainQuadrupedEnv with the 12-1024-512-8 policy;
  * gpu: the card's name and power limit, read by the same process.
Needs a CUDA device; there is no CPU fallback."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def _time(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="4096,16384,65536")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--horizon", type=int, default=24)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--collects", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_policy_wide.py needs a CUDA device")
    from opendog_b200.compat import BatchedQuadrupedEnv, BatchedTerrainQuadrupedEnv
    from opendog_b200.policy import ActorCriticB200
    from opendog_b200.rollout import Rollout
    res = {"gpu": _gpu_info(), "forward_ms": {}, "collect_ms_per_step": {}}
    pol = ActorCriticB200(12, 8, 0.3, hidden=(1024, 512), seed=1)
    for n in (int(x) for x in args.rows.split(",")):
        obs = torch.randn(n, 12, device="cuda")
        out = {k: torch.empty(n, 8, device="cuda") for k in ("mean", "action")}
        out.update({k: torch.empty(n, device="cuda") for k in ("value", "logp")})
        kern = _time(lambda: pol.act(obs, out=out, step=0), args.iters, 5)
        lib = _time(lambda: pol._act_library(obs, True, out), args.iters, 5)
        flop = 2 * n * 2 * (12 * 1024 + 1024 * 512) + 2 * n * 512 * 9
        res["forward_ms"][n] = {"kernel": round(kern, 4), "act_library": round(lib, 4),
                                "kernel_tflops": round(flop / kern / 1e9, 1)}
    for name, make, S, A, hidden in (("train_22-512-256-4", lambda n: BatchedQuadrupedEnv(n, auto_reset=True), 22, 4, (512, 256)),
                                     ("terrain_12-1024-512-8", lambda n: BatchedTerrainQuadrupedEnv(n, auto_reset=True), 12, 8, (1024, 512))):
        env = make(args.envs)
        p = ActorCriticB200(S, A, 0.4, hidden=hidden, seed=2)
        ro = Rollout(env, p, horizon=args.horizon, use_graph=True)
        ro.collect(); ro.collect()                           # eager warm-up, capture + first replay
        ms = _time(ro.collect, args.collects, 1)
        fwd = _time(lambda: p.act(ro.obs[0], step=0, out=dict(mean=ro.mean, value=ro.value[0], action=ro.action[0],
                                                               logp=ro.logp[0])), args.iters, 5)
        res["collect_ms_per_step"][name] = {"envs": args.envs, "horizon": args.horizon,
                                            "ms_per_policy_step": round(ms / args.horizon, 4),
                                            "policy_forward_ms": round(fwd, 4)}
        env.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
