#!/usr/bin/env python
"""bench.py — env-steps/s of the batched OpenDOG walk environment step on B200 (device-timed).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement on the host cores
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs (seeded inputs)

A "step" is one pass of the hot path over one batch: ONE Gym env-step (frame_skip = 10 physics
substeps, obs, reward, termination, auto-reset) of every environment of the batch. At N = 1 the
workload is BASELINE.json configs[1]: 4096 envs, OpenDOG MJCF, flat plane, PD actuators, fused
reward/obs/auto-reset. With N > 1 every rank steps its own shard of the same size (weak scaling, no
data-path collective; RNG streams keyed by global env id).

value      device-timed whole-job env-steps/s, actions already resident in HBM
e2e        same metric through BatchedWalkEnv.step with pinned HOST action buffers and a host read of
           (obs, reward, terminated, truncated) inside the timed region
roofline   HBM roofline of the step kernel: 542 algorithmic bytes per env-step (SURVEY §8d) x envs per
           launch / measured launch time, against MEASURED_PEAKS.json hbm_gbs. The kernel is FP32-ALU /
           latency bound, so the ALU fraction is reported next to it (roofline.alu).
cpu_baseline  the oracle port timed on the host cores on a bounded sample (rank 0, N = 1 only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
ALGO_BYTES_PER_ENV_STEP = 542          # SURVEY §8(d): 224 B read + 318 B write, fp32 SoA, walk/our_robot
FRAME_SKIP = 10
METRIC = "env-steps/sec (device-timed) at 1/2/4/8 B200 vs ref mj_step on host cores"


# ------------------------------------------------------------------------------------------- CPU arm
MUJOCO_SOLVER_DEFAULTS = dict(tolerance=1e-8, ls_tolerance=0.01, ls_iterations=50)     # mjOption defaults (mujoco 3.2.3)


def _cpu_worker(conn, n_envs, seed, first_id):
    """One worker = one host core stepping its own env set, like one SubprocVecEnv process (train/train.py:81-86), but
    with the whole set advanced by ONE C call per env-step (no per-env Python or ctypes overhead in the timed loop)."""
    import ctypes as C
    import numpy as np
    from oracle.oracle import WalkEnv, OdgoWalkEnv, lib
    L = lib()
    # stop the Newton solver where MuJoCo's defaults stop; the oracle's own (parity) setting is ~1000x tighter and would
    # make the CPU arm do several times the work mj_step does
    L.odgo_set_solver.argtypes = [C.c_double, C.c_double, C.c_int, C.c_int]
    L.odgo_set_solver(MUJOCO_SOLVER_DEFAULTS["tolerance"], MUJOCO_SOLVER_DEFAULTS["ls_tolerance"],
                      MUJOCO_SOLVER_DEFAULTS["ls_iterations"], 1)
    envs = [WalkEnv(seed=seed, env_id=first_id + i) for i in range(n_envs)]
    for e in envs:
        e.reset()
    ptrs = (C.POINTER(OdgoWalkEnv) * n_envs)(*[C.pointer(e.e) for e in envs])
    obs = np.zeros((n_envs, 33)); rew = np.zeros(n_envs); done = np.zeros(n_envs, np.int32)
    rng = np.random.default_rng(seed + first_id)
    fp = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg is None:
            break
        for _ in range(int(msg)):                        # msg = how many env-steps to advance before answering
            a = rng.uniform(-1, 1, (n_envs, 8)).astype(np.float32)
            L.odgo_walk_step_autoreset_batch(ptrs, n_envs, fp(a, C.c_float), fp(obs, C.c_double), fp(rew, C.c_double), fp(done, C.c_int))
        conn.send(n_envs * int(msg))
    conn.close()


class CpuPool:
    """`procs` OS processes, one oracle env set each — the layout of SB3 SubprocVecEnv (train/train.py:81-86)."""

    def __init__(self, total_envs, procs, seed=0):
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.procs, self.conns = [], []
        per = [total_envs // procs + (1 if i < total_envs % procs else 0) for i in range(procs)]
        first = 0
        for n in per:
            if n == 0:
                continue
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(b, n, seed, first), daemon=True)
            p.start()
            self.procs.append(p); self.conns.append(a)
            first += n
        for c in self.conns:
            c.recv()
        self.total = total_envs

    def step(self, count=1):
        for c in self.conns:
            c.send(count)
        return sum(c.recv() for c in self.conns)

    def close(self):
        for c in self.conns:
            c.send(None)
        for p in self.procs:
            p.join(timeout=5)


def cpu_throughput(sample_envs, steps, warmup, procs, chunk=1):
    """`steps` env-steps of every sample env, `chunk` of them per message to the workers."""
    pool = CpuPool(sample_envs, procs)
    for _ in range(warmup):
        pool.step()
    t0 = time.perf_counter()
    n = 0
    for _ in range(max(1, steps // chunk)):
        n += pool.step(chunk)
    dt = time.perf_counter() - t0
    pool.close()
    return n / dt, dt


REFERENCE_ENV_STEPS_PER_STEP = 30     # --impl reference: one bench "step" advances every sample env by this many env-steps


def cpu_baseline(all_core_steps, one_core_steps, envs_per_core=16, warmup=12, chunk=1):
    """The CPU arm on a bounded sample: all host cores (one process per core), then one core alone (SURVEY section 8d
    config 1 asks for both). Returns the `cpu_baseline` object of the bench line."""
    from oracle.oracle import build
    build()
    procs = os.cpu_count() or 1
    v_all, dt_all = cpu_throughput(procs * envs_per_core, all_core_steps, warmup, procs, chunk)
    v_one, dt_one = cpu_throughput(envs_per_core, one_core_steps, warmup, 1, chunk)
    return {"value": v_all, "unit": "env-steps/s", "cores": procs, "kind": "port",
            "one_core": {"value": v_one, "unit": "env-steps/s", "physics_steps_per_s": v_one * FRAME_SKIP},
            "physics_steps_per_s_per_core": v_all * FRAME_SKIP / procs,
            "solver": dict(MUJOCO_SOLVER_DEFAULTS, note="MuJoCo's default stopping rules; the parity oracle itself runs 1000x tighter"),
            "build": "gcc -O3 -march=native -ffp-contract=off, one C call per worker per env-step",
            "sample": f"all cores: {procs} processes x {envs_per_core} envs x {all_core_steps} env-steps ({dt_all:.1f} s); one core: "
                      f"{envs_per_core} envs x {one_core_steps} env-steps ({dt_one:.1f} s); after {warmup} warm-up env-steps (robots "
                      "landed). fp64 restatement of mj_step + the reference's reward code — NOT MuJoCo itself: mujoco==3.2.3 is "
                      "not installable here or on the GPU box (profiles/r02_mujoco_probe.txt)"}, dt_all


def workload_config(envs_per_gpu):
    """The `config` object of BOTH arms (ours and --impl reference): the workload and the timing rules, no measured values —
    so the two lines name the same configuration key for key. Arm-specific facts sit next to it (`physics_steps_per_s`,
    `solver`, `cpu_baseline.sample`)."""
    return {"workload": workload_name(envs_per_gpu), "envs_per_gpu": envs_per_gpu, "frame_skip": FRAME_SKIP,
            "l2": "GPU arm: flushed (256 MiB memset) between timed steps, per-step CUDA events summed; CPU arm: host caches, wall clock",
            "actions": "U(-1,1), a fresh batch every step (GPU arm: pre-generated on the device; CPU arm: drawn in each worker)",
            "cpu_arm": "every step advances a bounded sample of the workload (cpu_baseline.sample; with --impl reference by "
                       f"{REFERENCE_ENV_STEPS_PER_STEP} env-steps per env); throughput per env-step is what is compared"}


def workload_name(envs_per_gpu):
    return (f"{envs_per_gpu} envs/GPU batched step, OpenDOG MJCF (our_robot), flat-plane foot contact, PD "
            "position actuators, fused reward/obs/auto-reset (BASELINE.json configs[1])")


def run_reference(args):
    """CPU arm: the oracle restatement (the reference's mujoco wheel is not installable here) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # bounded sample: each "step" advances 16 envs per core by REFERENCE_ENV_STEPS_PER_STEP env-steps (a 4096-env batch would
    # cost ~0.09 s x 4096/16/cores per env-step). Several seconds of steady-state stepping whatever --steps is: a 0.2 s
    # sample right after the warm-up read 30 % low (round 2), which would flatter the GPU arm
    R = REFERENCE_ENV_STEPS_PER_STEP
    K = max(1, args.steps)
    cb, dt = cpu_baseline(all_core_steps=K * R, one_core_steps=min(K * R, 600), warmup=max(args.warmup, 12), chunk=R)
    value = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(ENVS_PER_GPU), "physics_steps_per_s": value * FRAME_SKIP,
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------- GPU arm
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nme in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def run_gpu(args):
    import numpy as np
    import torch
    from opendog_b200.env import BatchedWalkEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — opendog_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    N = args.envs_per_gpu
    K, W = args.steps, max(args.warmup, 3)
    SETTLE = 12          # untimed env-steps before anything is measured, whatever --warmup says: the reset drops the robots
                         # 0.13 m (~8 env-steps of free fall, then the landing transient); timed steps are stance / impact physics
    extra = {}
    for kv in args.cfg:
        k, v = kv.split("=")
        extra[k] = float(v) if "." in v or "e" in v else int(v)
    env = BatchedWalkEnv(N, device=dev, seed=0, first_env_id=rank * N, info_keys=None, **extra)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    # synthetic inputs: a fresh U(-1,1) action batch per step, generated on the device OUTSIDE the timed region
    actions = torch.rand(SETTLE + W + K, N, 8, device=dev, generator=gen) * 2 - 1
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local)
    sampler.start()
    for i in range(SETTLE):
        env.step(actions[i])
    actions = actions[SETTLE:]
    for i in range(W):                               # warm-up proper (same code path as the timed steps)
        flush.zero_()
        env.step(actions[i])
    barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    launches0 = env.launch_count
    import gc
    gc.collect()
    gc.disable()                                     # no collector pauses between the launches of the timed region
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(K):
        flush.zero_()                                # evict L2 between timed steps (not timed)
        starts[i].record()
        out = env.step(actions[W + i])
        ends[i].record()
    barrier()
    wall = time.perf_counter() - t_wall0
    launches = env.launch_count - launches0
    if args.dump_outputs:
        # copied now: obs and reward are views of the env's output buffer, which the e2e steps below overwrite
        obs, rew, done, _ = out
        dump_outputs(args.dump_outputs, {"obs": obs, "reward": rew, "done": done}, rank, world)
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    # ---- e2e: host buffers in, host results out, every step
    h_act = torch.empty(N, 8, pin_memory=True)
    h_obs = torch.empty(N, env.obs_dim, pin_memory=True)
    h_rew = torch.empty(N, pin_memory=True)
    h_term = torch.empty(N, dtype=torch.uint8, pin_memory=True)
    h_trunc = torch.empty(N, dtype=torch.uint8, pin_memory=True)
    d_act = torch.empty(N, 8, device=dev)
    host_actions = actions[W:W + K].cpu().pin_memory()      # the step's inputs wait in page-locked host memory (bench contract)
    e2e_steps = K
    for i in range(min(10, K)):                      # untimed: pinned-buffer allocation of step_host, host caches warm
        env.step_host(host_actions[i])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        # the reference-facing call with HOST buffers: fresh host action batch in (H2D), host obs / reward / terminated /
        # truncated out (D2H), synchronised — the caller reads the results before acting again
        h_obs, h_rew, h_term, h_trunc = env.step_host(host_actions[i])
    e1.record()
    barrier()
    gc.enable()
    e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    # ---- max over ranks
    t = torch.tensor([dev_ms, e2e_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    total_envs = N * world
    value = total_envs * K / (dev_ms * 1e-3)
    e2e_value = total_envs * e2e_steps / (e2e_ms * 1e-3)
    hbm_peak, peak_src, sm_max = measured_peaks()
    launch_s = dev_ms * 1e-3 / K
    achieved = ALGO_BYTES_PER_ENV_STEP * N / launch_s / 1e9
    # FP32 instruction-issue roofline: 148 SMs x 128 lanes x clock; ~6.4e5 lane-instructions per env-step (DESIGN.md)
    alu_peak_lane_ips = 148 * 128 * (clocks.get("sm_mhz") or sm_max) * 1e6
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W, "settle_steps": SETTLE,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(N), "physics_steps_per_s": value * FRAME_SKIP,
        "solver": {"max_newton_iters": env.cfg.solver_iterations, "ls_iters": env.cfg.ls_iterations, "tol": env.cfg.solver_tolerance},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": None, "peak_source": peak_src,
                     "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP,
                     "note": "state is reused across 10 substeps in registers: the kernel is FP32-issue/latency "
                             "bound, not HBM bound (see alu)",
                     "alu": {"lane_instr_per_s_peak": alu_peak_lane_ips}},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": N * 8 * 4,
                "d2h_bytes_per_step": int(env._out_bytes), "ms_per_step": e2e_ms / e2e_steps,
                "transfer": ("copy-engine H2D + D2H", "actions read in place from page-locked memory, D2H copy of the results",
                             "actions read from and results written to page-locked host memory by the kernel itself")[env.host_zero_copy]},
        "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": wall,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"], _ = cpu_baseline(all_core_steps=1200, one_core_steps=600)
    if rank == 0 and args.large_batch and world == 1:
        line["large_batch"] = large_batch_probe(dev, args.large_batch, extra)
    if rank == 0 and args.go1 and world == 1:
        line["step_go1"] = large_batch_probe(dev, N, None, model="go1")
    tr = profile_traffic(N)
    if tr:
        line["roofline"]["traffic"] = tr[0]
        line["roofline"]["traffic_source"] = f"profiles/{tr[1]} (ncu dram__bytes_read.sum + dram__bytes_write.sum, one launch)"
        if tr[3]:
            # FP32 roofline with COUNTED work (SURVEY section 8d ii): thread-level 2 x FFMA + FADD + FMUL of one launch
            # (ncu smsp__sass_thread_inst_executed_op_{ffma,fadd,fmul}_pred_on) / live launch time, against
            # 148 SMs x 128 lanes x 2 flop x SM clock under load
            clk = (clocks.get("sm_mhz") or sm_max) * 1e6
            peak = 148 * 128 * 2 * clk / 1e12
            ach = float(tr[3]) / launch_s / 1e12
            line["roofline"]["fp32"] = {"bound": "fp32", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                                        "counted_flops_per_launch": float(tr[3]), "counted_flops_per_env_step": float(tr[3]) / N,
                                        "sm_clock_mhz": clk / 1e6}
        if tr[2]:
            # issue-slot view of the same launch: warp-instructions per launch (ncu) / live launch time vs 4 issue slots
            # per SM per cycle. This, not HBM, is the resource the kernel is bound by (DESIGN.md section 4).
            peak_ips = 148 * 4 * (clocks.get("sm_mhz") or sm_max) * 1e6
            ach = float(tr[2]) / launch_s
            line["roofline"]["alu"] = {"bound": "issue", "warp_instructions_per_launch": float(tr[2]), "achieved": ach,
                                       "peak": peak_ips, "unit": "warp-inst/s", "frac": ach / peak_ips}
    if rank == 0 and world == 1 and args.mppi:
        line["mppi"] = mppi_probe(dev)
    if args.rollout_envs and (world > 1 or rank == 0):
        del env
        if world == 1:
            # BASELINE.json configs[2]: 16384 envs x horizon 24 with the policy on tensor cores, one GPU
            line["rollout"] = rollout_probe(dev, args.rollout_envs, args.horizon, rank, world, dist, train=args.train_probe)
        if args.train_envs:
            # BASELINE.json configs[3] as first-class keys at EVERY N (the timed `value` above is the collective-free
            # configs[1] step): 65536 envs per GPU, on-device rollout, GAE + advantage-statistics all-reduce, one PPO epoch
            # with a flat-gradient all-reduce per minibatch. Weak scaling: efficiency at N = value(N) / (N x value(1)).
            r = rollout_probe(dev, args.train_envs, args.horizon, rank, world, dist, train=True, iters=args.train_iters)
            if world > 1:
                line["rollout"] = r
            line["configs3"] = {
                "workload": f"{args.train_envs} envs/GPU x horizon {args.horizon} on {world} GPU(s) (BASELINE.json configs[3])",
                "rollout_env_steps_per_s": r["env_steps_per_s_rollout"],
                "train_iteration_env_steps_per_s": r["env_steps_per_s_train_iteration"],
                "train_iteration_env_steps_per_s_median_iteration": r["env_steps_per_s_train_iteration_median"],
                "ms_rollout": r["ms_per_rollout"], "ms_gae_and_stats_allreduce": r["ms_gae_and_stats_allreduce"],
                "ms_ppo_epoch": r["ms_ppo_epoch_with_grad_allreduce"],
                "ms_grad_allreduce": r["ms_grad_allreduce_per_iteration"], "grad_allreduce": r["grad_allreduce"],
                "ms_each_iteration": r["ms_each_iteration_this_rank"],      # [rollout, gae, ppo epoch] of every timed iteration, rank 0
                "ms_host": r.get("ms_host_in_ppo_call_each_iteration"),
                "ppo_update": r["ppo_update"], "scaling": "weak"}
        if world == 1 and args.go1:
            # BASELINE.json configs[2] names the 12-actuator model: Unitree Go1 through the same kernels (48-512-256-12)
            line["rollout_go1"] = rollout_probe(dev, args.rollout_envs, args.horizon, rank, world, dist, model="go1")
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, rank, world):
    """Write what the last timed step returned as `<name>.npy` in float32 (`<name>.rank<r>.npy` with several ranks), so
    that two builds can be compared output for output. Above DUMP_MAX_BYTES a fixed, seeded sample of environments is
    written, with their indices in `env_index.npy`."""
    import numpy as np
    import torch
    arrays = {k: v.detach().to("cpu", torch.float32).numpy() for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes for a in arrays.values()) // n
    budget = DUMP_MAX_BYTES - 4096                   # room for the .npy headers
    if n * row_bytes > budget:
        idx = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    suffix = f".rank{rank}" if world > 1 else ""
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}{suffix}.npy"), a)


def large_batch_probe(dev, n_envs, extra=None, model="our_robot"):
    """Throughput at the batch size of BASELINE.json configs[3] (65536 envs/GPU), same timing hygiene; with
    model="go1": the 12-actuator model of configs[1]/[2] at the headline batch size."""
    import torch
    from opendog_b200.env import BatchedWalkEnv
    env = BatchedWalkEnv(n_envs, model=model, device=dev, seed=0, info_keys=None, **(extra or {}))
    env.reset()
    acts = torch.rand(32, n_envs, env.act_dim, device=dev) * 2 - 1
    for i in range(20):                              # (robots dropped from the keyframe have landed, episodes are mixed)
        env.step(acts[i])
    torch.cuda.synchronize(dev)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(20, 32):
        env.step(acts[i])
    e.record()
    torch.cuda.synchronize(dev)
    ms = s.elapsed_time(e) / 12
    return {"envs": n_envs, "model": model, "obs_dim": env.obs_dim, "act_dim": env.act_dim, "ms_per_step": ms,
            "env_steps_per_s": n_envs / (ms * 1e-3),
            "note": "12 distinct action batches back to back after 20 warm-up steps; not L2-flushed (state + outputs stream through HBM "
                    "only once per step either way)"}


def profile_traffic(n_envs):
    """DRAM bytes per k_step launch from the newest committed ncu summary for this batch size (profiles/*.json)."""
    import glob
    best = None
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", f"*_k_step_{n_envs}.json"))):
        try:
            d = json.load(open(f))
            t = d["kernels"][0].get("dram_traffic_bytes")
            if t:
                best = (float(t), os.path.basename(f), d["kernels"][0].get("smsp__inst_executed.sum"),
                        d["kernels"][0].get("fp32_flops_per_launch"))
        except Exception:
            pass
    return best


def mppi_probe(dev, samples=1024, horizon=64):
    """BASELINE.json configs[4]: MPPI, 1024 samples x horizon 64 from a shared state, cost reduction on device."""
    import torch
    from opendog_b200.mppi import MPPI
    m = MPPI(samples, horizon, sigma=0.3, lam=1.0, seed=0, device=dev, use_graph=True)
    q = torch.tensor(m.env.desc["key_qpos"], dtype=torch.float32); q[2] = 0.075
    m.set_start(q, torch.zeros(m.env.nv))
    for _ in range(3):
        m.plan()
    torch.cuda.synchronize(dev)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 5
    s.record()
    for _ in range(iters):
        m.plan()
    e.record()
    torch.cuda.synchronize(dev)
    ms = s.elapsed_time(e) / iters
    return {"workload": f"{samples} samples x horizon {horizon}, shared start state, sigma 0.3, CUDA graph replay",
            "ms_per_plan": ms, "env_steps_per_s": samples * horizon / (ms * 1e-3), "plans_per_s": 1e3 / ms,
            "kernels_per_plan": m.kernels_per_plan, "min_cost": float(m.stats[0]), "mean_cost": float(m.stats[1])}


def rollout_probe(dev, n_envs, horizon, rank, world, dist, train=False, model="our_robot", iters=3):
    """BASELINE.json configs[2]/[3]: on-device PPO rollout (policy MLP on tensor cores + fused env step, one CUDA
    graph per horizon), GAE, and — with `train` — the advantage-statistics all-reduce and one PPO epoch with a flat
    gradient all-reduce per minibatch. Device-timed, max over ranks."""
    import torch
    from opendog_b200.env import BatchedWalkEnv
    from opendog_b200.policy import ActorCriticB200
    from opendog_b200.rollout import Rollout
    from opendog_b200.train import GraphedPPOUpdate, allreduce_flat_grads
    import gc
    torch.manual_seed(0)
    # objects of earlier probes (CUDA graphs, their private memory pools) die when Python's cycle collector gets round to
    # them; if that happens inside a timed iteration, the cudaFree calls stall the host between two graph launches and the
    # device idles (seen as one 40-500 ms "PPO epoch" among 14.5 ms ones). Collect now, and keep the collector off while timing.
    gc.collect()
    torch.cuda.empty_cache()
    env = BatchedWalkEnv(n_envs, model=model, device=dev, seed=0, first_env_id=rank * n_envs, info_keys=None)
    pol = ActorCriticB200(env.obs_dim, env.act_dim, 0.4, device=dev, seed=0)
    ro = Rollout(env, pol, horizon=horizon, use_graph=True, first_row_id=rank * n_envs)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    def sync():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)
    opt = torch.optim.Adam(pol.parameters(), lr=1e-4, fused=True, capturable=True)
    T, N = ro.T, n_envs
    # the PPO epoch (4 minibatches: forward, loss, backward, flat-gradient all-reduce, clipping, fused Adam) is captured
    # once as CUDA graphs and replayed: no launch / allocator / lazy-loading time inside the timed iterations
    upd = GraphedPPOUpdate(pol, opt, T * N, env.obs_dim, env.act_dim, minibatches=4) if train else None
    for w in range(5):
        ro.collect()
        if w >= 1:                       # untimed, four times: first-use costs of the collectives, autograd and cuBLAS, graph capture
            adv, ret, stats = ro.advantages(normalize=True)
            if train:
                upd(ro.obs[:T].reshape(T * N, -1), ro.action.reshape(T * N, -1), ro.logp.reshape(-1), adv.reshape(-1), ret.reshape(-1))
    gc.collect()
    gc.disable()
    sync()
    # No host synchronisation inside the timed iterations (a training loop has none either): the host enqueues an iteration
    # while the device is still busy with the previous one, so a late host — on ANY rank: every rank waits for the
    # slowest one in the epoch's first all-reduce — costs nothing unless it is later than the ~100 ms of queued work.
    E = [[ev() for _ in range(4)] for _ in range(iters)]
    t_roll = t_gae = t_upd = t_ar = 0.0
    each = []
    host_ms = []
    for it in range(iters):
        e = E[it]
        e[0].record(); ro.collect(); e[1].record()
        adv, ret, stats = ro.advantages(normalize=True)       # all-reduces [sum, sumsq, n] when world > 1
        e[2].record()
        h0 = time.perf_counter()
        if train:
            upd(ro.obs[:T].reshape(T * N, -1), ro.action.reshape(T * N, -1), ro.logp.reshape(-1), adv.reshape(-1), ret.reshape(-1))
        h1 = time.perf_counter()
        e[3].record()
        host_ms.append((h1 - h0) * 1e3)
    torch.cuda.synchronize(dev)
    for e in E:
        t_roll += e[0].elapsed_time(e[1]); t_gae += e[1].elapsed_time(e[2]); t_upd += e[2].elapsed_time(e[3])
        each.append([e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2]), e[2].elapsed_time(e[3])])
    gc.enable()
    e = E[0]
    if train:
        # the flat-gradient all-reduce alone (the captured epoch contains 4 of them): same buffer, same collective
        params = [p for p in pol.parameters() if p.requires_grad]
        for _ in range(2):
            allreduce_flat_grads(params)
        sync()
        ea = [ev(), ev()]
        ea[0].record()
        for _ in range(4 * iters):
            allreduce_flat_grads(params)
        ea[1].record()
        torch.cuda.synchronize(dev)
        t_ar = ea[0].elapsed_time(ea[1])
    # the policy forward alone (same launches as inside the rollout)
    l0 = pol.launch_count
    e[0].record()
    for t in range(horizon + 1):
        pol.act(ro.obs[min(t, horizon)], sample=True, step=t, out=dict(mean=ro.mean, value=ro.value[t], action=ro.action[min(t, horizon - 1)], logp=ro.logp[min(t, horizon - 1)]))
    e[1].record()
    torch.cuda.synchronize(dev)
    t_mlp = e[0].elapsed_time(e[1]) / (pol.launch_count - l0)
    t = torch.tensor([t_roll, t_gae, t_upd, t_mlp, t_ar], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_roll, t_gae, t_upd, t_mlp, t_ar = [float(x) for x in t]
    S, A = env.obs_dim, env.act_dim
    flops = 2.0 * (S * 512 + 512 * 256 + 256 * A) + 2.0 * (S * 512 + 512 * 256 + 256)      # actor + critic, per env
    pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    peak = float(pk.get("bf16_tflops_sustained", 1400.0))
    ach = flops * n_envs / (t_mlp * 1e-3) / 1e12
    steps = n_envs * world * horizon * iters
    out = {"workload": f"{n_envs} envs/GPU x horizon {horizon}, model {model}, ActorCritic {S}-512-256-{A} (+critic) bf16 tcgen05, CUDA graph",
           "env_steps_per_s_rollout": steps / (t_roll * 1e-3), "ms_per_rollout": t_roll / iters,
           "ms_gae_and_stats_allreduce": t_gae / iters, "ms_policy_forward": t_mlp,
           "policy_share_of_rollout": t_mlp * (horizon + 1) / (t_roll / iters),
           "policy_roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                               "flops_per_env": flops, "note": "three skinny layers (K = 48/512/256) fused per 128-env CTA; weight streaming from L2 bound"},
           "kernels_per_rollout": ro.kernels_per_collect}
    if train:
        n_param = sum(p.numel() for p in pol.parameters())
        out["ms_ppo_epoch_with_grad_allreduce"] = t_upd / iters
        out["ms_each_iteration_this_rank"] = [[round(x, 3) for x in row] for row in each]      # [rollout, gae, ppo] x iterations
        out["ms_host_in_ppo_call_each_iteration"] = [round(x, 3) for x in host_ms]   # host time spent inside the (asynchronous) update call: enqueue only
        out["ms_grad_allreduce_per_iteration"] = t_ar / iters
        out["grad_allreduce"] = {"calls_per_iteration": 4, "payload_bytes_per_call": 4 * n_param,
                                 "ms_per_call": t_ar / iters / 4,
                                 "share_of_train_iteration": t_ar / max(t_roll + t_gae + t_upd, 1e-9),
                                 "note": "flat fp32 gradient buffer (pack + NCCL all-reduce + unpack), timed alone right after the iterations (inside them it is part of the captured epoch)"}
        out["ppo_update"] = "1 epoch x 4 minibatches replayed as CUDA graphs: bf16 autocast forward/backward (fp32 master weights), flat-gradient all-reduce, clipping, fused Adam"
        out["env_steps_per_s_train_iteration"] = steps / ((t_roll + t_gae + t_upd) * 1e-3)
        # the same from the MEDIAN iteration of this rank (an iteration in which one rank's host starts its rollout late shows up
        # on every other rank as time spent waiting in the epoch's first all-reduce: ms_each_iteration)
        med = sorted(sum(row) for row in each)[len(each) // 2]
        out["env_steps_per_s_train_iteration_median"] = n_envs * world * horizon / (med * 1e-3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--large-batch", type=int, default=65536, help="also probe this batch size at N=1 (0 = off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rollout-envs", type=int, default=16384, help="N=1: also time the on-device PPO rollout (0 = off)")
    ap.add_argument("--train-envs", type=int, default=65536, help="N>1: envs per GPU of the train-iteration probe")
    ap.add_argument("--horizon", type=int, default=24)
    ap.add_argument("--train-iters", type=int, default=5, help="timed iterations of the train-iteration probe")
    ap.add_argument("--go1", type=int, default=1, help="N=1: also time the rollout on the 12-actuator Go1 model; 0 = off")
    ap.add_argument("--mppi", type=int, default=1, help="N=1: also time one MPPI plan (1024 x 64); 0 = off")
    ap.add_argument("--train-probe", action="store_true", help="N=1: include the PPO epoch in the rollout probe")
    ap.add_argument("--cfg", action="append", default=[], help="OdgEnvConfig override key=value (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's obs / reward / done to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
