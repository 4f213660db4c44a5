"""Sampling-MPC (MPPI) on the batched simulator: BASELINE.json configs[4] — `num_samples` action sequences of length
`horizon` rolled out from ONE shared robot state, costs reduced on the device (include/odg_mppi.h). The reference has
no MPC code; the cost is minus the reference's walk reward (WalkEnvironment.py:81-109, taken BEFORE its max(0, .)
clip, which would zero most of the signal) summed along the rollout.

Per plan(): broadcast the start state, ONE rollout launch (`odg_mppi_rollout`: every sample walks its whole horizon —
sample the action row, fused env step, accumulate the cost — without leaving the SM) and one reduction launch
(`odg_mppi_reduce`). The plan counter that keys the noise lives in device memory and is incremented on the stream, so
a captured CUDA graph draws fresh noise on every replay.

`BatchedMPPI` plans for K robots of a `BatchedWalkEnv` at once, each from its own state, and runs the closed MPC loop
on the device (`control_step`).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import lib as _lib
from .env import BatchedWalkEnv, _ptr


class MPPI:
    def __init__(self, num_samples: int = 1024, horizon: int = 64, sigma: float = 0.3, lam: float = 1.0,
                 termination_cost: float = 100.0, device=None, seed: int = 0, use_graph: bool = True, **sim_config):
        self.env = BatchedWalkEnv(num_samples, device=device, seed=seed, info_keys=None, auto_reset=0, **sim_config)
        self.L, self.dev = self.env.L, self.env.device
        self.N, self.T, self.A = num_samples, horizon, self.env.act_dim
        self.sigma, self.lam, self.term_cost, self.seed = sigma, lam, termination_cost, seed
        dev = self.dev
        self.mean = torch.zeros(horizon, self.A, device=dev)               # nominal sequence (actions in [-1, 1])
        self.new_mean = torch.zeros(horizon, self.A, device=dev)
        self.actions = torch.zeros(horizon, num_samples, self.A, device=dev)
        self.cost = torch.zeros(num_samples, device=dev)
        self.stats = torch.zeros(4, device=dev)
        # shared start state, broadcast to every sample at the start of a plan
        self.q0 = torch.zeros(num_samples, self.env.nq, device=dev)
        self.v0 = torch.zeros(num_samples, self.env.nv, device=dev)
        self.env_state0 = None
        self.iteration = 0
        self.iteration_dev = torch.zeros(1, dtype=torch.int32, device=dev)     # plan counter keying the noise (Philox)
        self.use_graph, self.graph = use_graph, None

    def _st(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def set_start(self, qpos, qvel, last_action=None, desired_velocity=None):
        """The shared robot state: qpos [nq], qvel [nv] (+ the env-side state the walk reward reads)."""
        self.q0.copy_(torch.as_tensor(qpos, dtype=torch.float32).to(self.dev).reshape(1, -1).expand(self.N, -1))
        self.v0.copy_(torch.as_tensor(qvel, dtype=torch.float32).to(self.dev).reshape(1, -1).expand(self.N, -1))
        la = torch.zeros(self.A) if last_action is None else torch.as_tensor(last_action, dtype=torch.float32)
        dv = torch.tensor([0.75, 0.0, 0.0]) if desired_velocity is None else torch.as_tensor(desired_velocity, dtype=torch.float32)
        z = torch.zeros(self.N, dtype=torch.int32)
        self.env_state0 = dict(step=z.to(self.dev), gait_index=z.to(self.dev), gait_matches=z.to(self.dev),
                               last_action=la.reshape(1, -1).expand(self.N, -1).contiguous().to(self.dev),
                               desired_velocity=dv.reshape(1, -1).expand(self.N, -1).contiguous().to(self.dev),
                               fresh=torch.zeros(self.N, dtype=torch.uint8, device=self.dev))

    def _body(self):
        e, L, st = self.env, self.L, self._st()
        _lib.check(L.odg_set_state(e._h, _ptr(self.q0), _ptr(self.v0), None, st), "odg_set_state")
        s0 = self.env_state0
        _lib.check(L.odg_set_env_state(e._h, _ptr(s0["step"]), _ptr(s0["gait_index"]), _ptr(s0["gait_matches"]),
                                       _ptr(s0["last_action"]), _ptr(s0["desired_velocity"]), _ptr(s0["fresh"]), st),
                   "odg_set_env_state")
        _lib.check(L.odg_mppi_rollout(e._h, _ptr(self.mean), self.sigma, self.T, C.c_uint64(self.seed), 0, _ptr(self.iteration_dev),
                                      self.term_cost, _ptr(self.actions), _ptr(self.cost), st), "odg_mppi_rollout")
        _lib.check(L.odg_mppi_reduce(_ptr(self.cost), _ptr(self.actions), self.T, self.N, self.A, self.lam,
                                     _ptr(self.new_mean), _ptr(self.stats), st), "odg_mppi_reduce")
        self.iteration_dev.add_(1)

    def plan(self, update_mean: bool = True):
        """One MPPI iteration from the shared start state; returns the updated nominal sequence [T, A]."""
        assert self.env_state0 is not None, "call set_start first"
        if not self.use_graph:
            self._body()
        elif self.graph is not None:
            self.graph.replay()
        elif self.iteration == 0:
            self._body()                 # first plan runs eagerly: it is also the warm-up the capture needs
        else:
            torch.cuda.synchronize(self.dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._body()
            self.graph.replay()          # capture only records: run it once
        self.iteration += 1
        if update_mean:
            self.mean.copy_(self.new_mean)
        return self.new_mean

    @property
    def kernels_per_plan(self) -> int:
        return 9          # 2 + 5 state-broadcast transposes / copies, the rollout, the reduction, the counter


class BatchedMPPI:
    """MPPI for K robots at once, each planned from its own state: K groups of `samples_per_robot` samples in one samples
    environment (include/odg_mppi.h, "Batched MPPI"). Group g follows the nominal sequence `mean[g]` and draws the noise
    of a single-robot plan with seed `seed + g`, so it equals that plan bit for bit.

    `robots` is the batch being controlled; robots [first_robot, first_robot + num_robots) are planned (default: all).
    The samples environment has the robots' model and every `OdgEnvConfig` field of `robots.cfg` except `auto_reset`,
    which is 0. Per plan(): `odg_mppi_broadcast` (each robot's full state, warm start included, into its group),
    `odg_mppi_rollout_groups` (one launch) and `odg_mppi_reduce_groups` (one block per robot), then the plan counter is
    bumped on the device. `control_step()` closes the loop on the device: plan, step the robots with the first action
    of each new nominal sequence, shift the sequences and zero those of robots whose episode ended.
    With `use_graph`, the first call of `plan` / `control_step` runs eagerly (warm-up), the second captures a CUDA graph
    and later calls replay it.
    """

    def __init__(self, robots: BatchedWalkEnv, samples_per_robot: int = 1024, horizon: int = 64, sigma: float = 0.3,
                 lam: float = 1.0, termination_cost: float = 100.0, seed: int = 0, use_graph: bool = True,
                 num_robots: int | None = None):
        self.robots = robots
        self.K = robots.num_envs if num_robots is None else int(num_robots)
        if not 1 <= self.K <= robots.num_envs:
            raise ValueError(f"num_robots must be in [1, {robots.num_envs}]")
        self.S, self.T, self.A = int(samples_per_robot), int(horizon), robots.act_dim
        cfg = {name: getattr(robots.cfg, name) for name, _ in _lib.OdgEnvConfig._fields_}
        cfg["auto_reset"] = 0
        self.env = BatchedWalkEnv(self.K * self.S, model=robots.model, device=robots.device, seed=seed, info_keys=None, **cfg)
        self.L, self.dev = self.env.L, self.env.device
        self.sigma, self.lam, self.term_cost, self.seed = sigma, lam, termination_cost, seed
        K, T, A, dev = self.K, self.T, self.A, self.dev
        self.mean = torch.zeros(K, T, A, device=dev)                        # nominal sequences (actions in [-1, 1])
        self.new_mean = torch.zeros(K, T, A, device=dev)
        self.actions = torch.zeros(T, K * self.S, A, device=dev)
        self.cost = torch.zeros(K * self.S, device=dev)
        self.stats = torch.zeros(K, 4, device=dev)                          # per robot: min, mean cost, sum w, argmin
        self.action = torch.zeros(K, A, device=dev)                         # control_step: the robots' actions
        self._done = torch.zeros(K, dtype=torch.bool, device=dev)
        self.iteration = 0                                                  # plans so far (host-side count)
        self.iteration_dev = torch.zeros(1, dtype=torch.int32, device=dev)  # plan counter keying the noise (Philox)
        self.use_graph = use_graph
        self._graphs = {}                                                   # "plan" / "control" -> (CUDAGraph, first_robot)
        self._calls = {"plan": 0, "control": 0}

    def _st(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def _plan_body(self, first_robot: int):
        L, st, K = self.L, self._st(), self.K
        _lib.check(L.odg_mppi_broadcast(self.env._h, self.robots._h, first_robot, K, st), "odg_mppi_broadcast")
        _lib.check(L.odg_mppi_rollout_groups(self.env._h, K, _ptr(self.mean), self.sigma, self.T, C.c_uint64(self.seed), 0,
                                             _ptr(self.iteration_dev), self.term_cost, _ptr(self.actions), _ptr(self.cost), st),
                   "odg_mppi_rollout_groups")
        _lib.check(L.odg_mppi_reduce_groups(_ptr(self.cost), _ptr(self.actions), self.T, K, self.S, self.A, self.lam,
                                            _ptr(self.new_mean), _ptr(self.stats), st), "odg_mppi_reduce_groups")

    def _control_body(self):
        r = self.robots
        self._plan_body(0)
        self.action.copy_(self.new_mean[:, 0])
        r.step_into(self.action, r.obs, r.reward, r.terminated, r.truncated)
        self.mean[:, :-1].copy_(self.new_mean[:, 1:])
        self.mean[:, -1].zero_()
        torch.logical_or(r.terminated, r.truncated, out=self._done)
        self.mean.masked_fill_(self._done.view(-1, 1, 1), 0.0)             # an ended episode starts from a zero nominal

    def _run(self, kind: str, body, first_robot: int):
        if not self.use_graph:
            body()
            return
        g = self._graphs.get(kind)
        if g is not None:
            if g[1] != first_robot:
                raise ValueError(f"the captured {kind} graph plans from first_robot = {g[1]}, not {first_robot}")
            g[0].replay()
        elif self._calls[kind] == 0:
            body()                       # the first call runs eagerly: it is also the warm-up the capture needs
        else:
            torch.cuda.synchronize(self.dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                body()
            self._graphs[kind] = (graph, first_robot)
            graph.replay()               # capture only records: run it once
        self._calls[kind] += 1

    def plan(self, first_robot: int = 0):
        """One MPPI iteration for robots [first_robot, first_robot + K) from their current states; returns the updated
        nominal sequences [K, T, A] (`mean` is left as it was)."""
        if not 0 <= first_robot <= self.robots.num_envs - self.K:
            raise ValueError(f"first_robot must be in [0, {self.robots.num_envs - self.K}]")

        def body():
            self._plan_body(first_robot)
            self.iteration_dev.add_(1)
        self._run("plan", body, first_robot)
        self.iteration += 1
        return self.new_mean

    def control_step(self):
        """One receding-horizon step for every robot, with no host synchronisation: plan; step the robots with
        new_mean[:, 0]; mean[:, :-1] <- new_mean[:, 1:], mean[:, -1] <- 0; zero the nominal of every robot whose step
        ended its episode (the robots' own auto-reset starts the next one); bump the plan counter. Returns the robots'
        (obs, reward, terminated, truncated) buffers."""
        if self.K != self.robots.num_envs:
            raise ValueError("control_step plans every robot: create BatchedMPPI without num_robots")

        def body():
            self._control_body()
            self.iteration_dev.add_(1)
        self._run("control", body, 0)
        self.iteration += 1
        r = self.robots
        return r.obs, r.reward, r.terminated, r.truncated
