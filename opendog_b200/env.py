"""Batched, GPU-resident environments behind the reference's Gym-style surface.

`BatchedWalkEnv` is `ScaleActionWrapper(WalkEnvironmentV0)` (reference:
Code/mujoco/environments/WalkEnvironment.py:26-158, ScaleActionEnvironment.py:5-23) for `num_envs`
environments at once: `reset()` / `step(action) -> (obs, reward, done, info)` on CUDA tensors, state
never leaves HBM. PyTorch only provides the device buffers and the stream; the work happens in
libodgsim's hand-written kernels through the C ABI (include/odg.h).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import lib as _lib
from .model.compile import load_compiled, to_struct

_INFO_SPECS = {
    # name in OdgInfoPtrs -> (dtype, trailing shape factory)
    "x_position": (torch.float32, lambda e: ()),
    "y_position": (torch.float32, lambda e: ()),
    "distance_from_origin": (torch.float32, lambda e: ()),
    "paw_contact_forces": (torch.float32, lambda e: (4, 6)),
    "patterns_matches": (torch.float32, lambda e: ()),
    "linear_vel_tracking_reward": (torch.float32, lambda e: ()),
    "reward_ctrl": (torch.float32, lambda e: ()),
    "terminal_obs": (torch.float32, lambda e: (e.obs_dim,)),
    "paws_in_ground": (torch.uint8, lambda e: (4,)),
    "gait_reward": (torch.int32, lambda e: ()),
    "qacc": (torch.float32, lambda e: (e.nv,)),
    "ncon": (torch.int32, lambda e: ()),
    "contact_normal_force": (torch.float32, lambda e: ()),
    "solver_iters": (torch.int32, lambda e: ()),
    "ls_evals": (torch.int32, lambda e: ()),
    "reward_unclipped": (torch.float32, lambda e: ()),
    # 12-actuator model (Go1): data.cfrc_ext[1:] and the jump task's weighted reward terms
    "cfrc_ext": (torch.float32, lambda e: (13, 6)),
    "task_terms": (torch.float32, lambda e: (10,)),
}
TASKS = {"walk": 0, "jump": 1}
JUMP_TERMS = ("landing_precision", "landing_orientation", "control_velocity_horizontal", "height_clearance", "phase_sync",
              "jump_velocity", "distance_on_liftoff", "vertical_velocity_on_landing", "out_of_bounds", "collision_cost")
DEFAULT_INFO = ("x_position", "y_position", "distance_from_origin", "paw_contact_forces", "patterns_matches",
                "linear_vel_tracking_reward", "reward_ctrl", "terminal_obs")


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class BatchedWalkEnv:
    """`num_envs` copies of the reference walk environment stepped by one fused CUDA kernel.

    Parameters mirror the reference's constants; see `OdgEnvConfig` in include/odg.h.
    `info_keys`: which `info` tensors `step` fills (None = none: fastest).
    """

    def __init__(self, num_envs: int, model: str = "our_robot", device=None, seed: int = 0,
                 info_keys=DEFAULT_INFO, **config):
        if not torch.cuda.is_available():
            raise _lib.OdgError("BatchedWalkEnv needs a CUDA device: opendog_b200 has no CPU fallback")
        self.L = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.model = model
        self.desc = load_compiled(model)
        self._model = to_struct(self.desc)
        self.cfg = _lib.OdgEnvConfig()
        self.L.odg_default_config(C.byref(self.cfg))
        if self.desc["nu"] == 12:
            self.cfg.obs_layout = 1        # 12-actuator models: the 48-value layout (landing_environment.py:116-136 + v_des)
        task = config.pop("task", "walk")
        # step_host: 0 = H2D copy of the actions and D2H copy of the output slab; 1 = the kernel reads the page-locked actions
        # in place over PCIe; 2 (default) = and writes obs / reward / terminated / truncated straight into the page-locked
        # result buffer (the info arrays too when the call asks for them). Same bits either way. Measured (tools/ab_e2e.py):
        # 4096 envs 0.445 -> 0.428 ms per step (with the default info arrays 0.466 -> 0.453), 16384 envs +-0, 65536 envs
        # 3.67 -> 3.54 ms (the results cross PCIe while the kernel's later tiles still run)
        self.host_zero_copy = int(config.pop("host_zero_copy", 2))
        self.cfg.task = TASKS[task] if isinstance(task, str) else int(task)
        if self.cfg.task == TASKS["jump"]:
            # JumpEnvironmentV0 is not wrapped in ScaleActionWrapper: actions are ctrl targets; its reward calculator's
            # reset_noise_scale is 0.1 (jump_environment_reward_calc.py:52)
            self.cfg.scale_actions = 0
            self.cfg.reset_noise_scale = 0.1
        for k, v in config.items():
            if not hasattr(self.cfg, k):
                raise TypeError(f"unknown config field {k!r}")
            setattr(self.cfg, k, v)
        self.num_envs = int(num_envs)
        h = C.c_void_p()
        _lib.check(self.L.odg_create(C.byref(self._model), C.byref(self.cfg), self.num_envs, self.device.index,
                                     C.c_uint64(seed), C.byref(h)), "odg_create")
        self._h = h
        self.obs_dim = self.L.odg_obs_dim(h)
        self.act_dim = self.L.odg_act_dim(h)
        self.nq, self.nv = self.L.odg_nq(h), self.L.odg_nv(h)
        self._host = None
        self.info = {}
        self._info_struct = None
        self.set_info_keys(info_keys)

    # ------------------------------------------------------------------ plumbing
    def set_info_keys(self, keys):
        """Choose the `info` tensors `step` fills and (re)allocate the output slab. Step outputs AND info tensors live in
        ONE device buffer — [obs | reward | terminated | truncated | info arrays...], every array 16-byte aligned — so a
        host-side caller fetches everything a step produced with a single device->host copy (`step_host`)."""
        N, dev = self.num_envs, self.device
        keys = tuple(keys or ())
        al = lambda n: (n + 15) // 16 * 16
        esz = {torch.float32: 4, torch.int32: 4, torch.uint8: 1}
        parts = [("obs", torch.float32, (N, self.obs_dim)), ("reward", torch.float32, (N,)),
                 ("terminated", torch.uint8, (N,)), ("truncated", torch.uint8, (N,))]
        for k in keys:
            dt, shp = _INFO_SPECS[k]
            parts.append((k, dt, (N,) + tuple(shp(self))))
        offs, o = [], 0
        for _, dt, shp in parts:
            offs.append(o)
            n = esz[dt]
            for d in shp:
                n *= d
            o += al(n)
        self._slab = torch.zeros(o, dtype=torch.uint8, device=dev)
        self._slab_layout = [(name, dt, shp, off) for (name, dt, shp), off in zip(parts, offs)]
        self._out_bytes = offs[4] if len(parts) > 4 else o          # bytes of the [obs | reward | flags] prefix
        views = {name: self._view(self._slab, dt, shp, off) for name, dt, shp, off in self._slab_layout}
        self.obs, self.reward = views["obs"], views["reward"]
        self.terminated, self.truncated = views["terminated"], views["truncated"]
        self._out = self._slab[:self._out_bytes]
        self._host = None
        self.info = {k: views[k] for k in keys}
        if not keys:
            self._info_struct = None
            return
        s = _lib.OdgInfoPtrs()
        for k in keys:
            setattr(s, k, self.info[k].data_ptr())
        self._info_struct = s

    @staticmethod
    def _view(buf, dt, shp, off):
        n = {torch.float32: 4, torch.int32: 4, torch.uint8: 1}[dt]
        for d in shp:
            n *= d
        return buf[off:off + n].view(dt).view(shp)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None):
            self.L.odg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self.L.odg_launch_count(self._h))

    # ------------------------------------------------------------------ Gym surface
    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        """env.reset() for all (or masked) envs; returns obs [N, obs_dim] (a view of an internal buffer)."""
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.L.odg_reset(self._h, _ptr(m), _ptr(self.obs), self._stream()), "odg_reset")
        return self.obs

    def step(self, action: torch.Tensor):
        """(obs, reward, done, info): `done = terminated | truncated`; with auto_reset the returned obs of
        a done env is its reset obs and info["terminal_obs"] holds the last obs of the episode."""
        self.step_into(action, self.obs, self.reward, self.terminated, self.truncated)
        done = (self.terminated | self.truncated).bool()
        return self.obs, self.reward, done, self.info

    def step_host(self, action_host: torch.Tensor, with_info: bool = False):
        """`step` for a caller whose policy lives on the HOST (SB3, the reference's loops): pinned host action in,
        pinned host (obs, reward, terminated, truncated) out — one H2D copy, one kernel, one D2H copy, one sync.
        With `with_info` the same single D2H copy also brings every `info` array (they share the slab) and a dict of
        host views is returned as a fifth element. The returned arrays are views of an internal pinned buffer, valid
        until the next call."""
        N = self.num_envs
        torch.cuda.nvtx.range_push("odg.step_host")
        try:
            return self._step_host(action_host, with_info, N)
        finally:
            torch.cuda.nvtx.range_pop()

    def _step_host(self, action_host, with_info, N):
        if self._host is None:
            h = torch.empty_like(self._slab, device="cpu").pin_memory()
            self._host = dict(slab=h, act=torch.empty(N, self.act_dim).pin_memory(),
                              dact=torch.empty(N, self.act_dim, device=self.device))
            for name, dt, shp, off in self._slab_layout:
                self._host[name] = self._view(h, dt, shp, off)
            # the call's fixed pointer arguments, built once (this method runs once per env-step of a host-side loop)
            self._host["args"] = (_ptr(self._host["act"]), _ptr(self._host["dact"]), _ptr(self.obs), _ptr(self.reward),
                                  _ptr(self.terminated), _ptr(self.truncated), _ptr(self._slab), _ptr(h))
            self._host["args_inplace"] = tuple(_ptr(self._host[k]) for k in ("obs", "reward", "terminated", "truncated"))
            self._host["info_inplace"] = None
            if self.info:
                hs = _lib.OdgInfoPtrs()                             # the same info arrays, in the page-locked slab
                for k in self.info:
                    setattr(hs, k, self._host[k].data_ptr())
                self._host["info_inplace"] = hs
        H = self._host
        a = action_host
        if a.device.type != "cpu" or a.dtype != torch.float32 or not a.is_contiguous():
            a = a.to(device="cpu", dtype=torch.float32).contiguous()
        if a.shape != (N, self.act_dim):
            raise ValueError(f"action must be [{N}, {self.act_dim}]")
        nb = self._slab.numel() if with_info else self._out_bytes
        info = C.byref(self._info_struct) if self._info_struct is not None else None
        # one C call: (memcpy to the page-locked staging buffer unless the caller's tensor is it) -> H2D -> step kernel ->
        # one D2H of the output slab -> stream synchronize (include/odg.h: odg_step_host)
        staged = a.data_ptr() == H["act"].data_ptr() or a.is_pinned()
        p_act, p_dact, p_obs, p_rew, p_term, p_trunc, p_slab, p_hslab = H["args"]
        if self.host_zero_copy >= 1:
            p_dact = _ptr(a) if staged else p_act                   # the kernel reads the page-locked actions in place
        if self.host_zero_copy >= 2:
            p_obs, p_rew, p_term, p_trunc = H["args_inplace"]       # ... and writes its results into the page-locked buffer
            if with_info and H["info_inplace"] is not None:
                info = C.byref(H["info_inplace"])
            p_slab = p_hslab = None
            nb = 0
        _lib.check(self.L.odg_step_host(self._h, _ptr(a), None if staged else p_act, p_dact, p_obs, p_rew, p_term, p_trunc, info,
                                        p_slab, p_hslab, nb, self._stream()), "odg_step_host")
        if with_info:
            return H["obs"], H["reward"], H["terminated"], H["truncated"], {k: H[k] for k in self.info}
        return H["obs"], H["reward"], H["terminated"], H["truncated"]

    def step_into(self, action: torch.Tensor, obs, reward, terminated, truncated):
        """`step` writing straight into caller-owned CUDA tensors (rollout buffers): no copies, no extra kernels."""
        a = action
        if a.device != self.device or a.dtype != torch.float32 or not a.is_contiguous():
            a = a.to(device=self.device, dtype=torch.float32).contiguous()
        if a.shape != (self.num_envs, self.act_dim):
            raise ValueError(f"action must be [{self.num_envs}, {self.act_dim}]")
        info = C.byref(self._info_struct) if self._info_struct is not None else None
        _lib.check(self.L.odg_step(self._h, _ptr(a), _ptr(obs), _ptr(reward), _ptr(terminated), _ptr(truncated), info,
                                   self._stream()), "odg_step")

    def evaluate(self, ctrl: torch.Tensor):
        """Test hook (odg_evaluate): one mj_forward on the current state + the post-step logic."""
        a = ctrl.to(device=self.device, dtype=torch.float32).contiguous()
        info = C.byref(self._info_struct) if self._info_struct is not None else None
        _lib.check(self.L.odg_evaluate(self._h, _ptr(a), _ptr(self.obs), _ptr(self.reward), _ptr(self.terminated),
                                       _ptr(self.truncated), info, self._stream()), "odg_evaluate")
        return self.obs, self.reward, self.terminated.bool(), self.truncated.bool(), self.info

    # ------------------------------------------------------------------ state access (parity tests)
    def get_state(self):
        qpos = torch.empty(self.num_envs, self.nq, device=self.device)
        qvel = torch.empty(self.num_envs, self.nv, device=self.device)
        _lib.check(self.L.odg_get_state(self._h, _ptr(qpos), _ptr(qvel), self._stream()), "odg_get_state")
        return qpos, qvel

    def set_state(self, qpos, qvel, qacc_warmstart=None):
        f = lambda t: None if t is None else torch.as_tensor(t, dtype=torch.float32).to(self.device).contiguous()
        qpos, qvel, w = f(qpos), f(qvel), f(qacc_warmstart)
        _lib.check(self.L.odg_set_state(self._h, _ptr(qpos), _ptr(qvel), _ptr(w), self._stream()), "odg_set_state")
        torch.cuda.current_stream(self.device).synchronize()

    def get_env_state(self):
        N, dev = self.num_envs, self.device
        o = dict(step=torch.empty(N, dtype=torch.int32, device=dev), gait_index=torch.empty(N, dtype=torch.int32, device=dev),
                 gait_matches=torch.empty(N, dtype=torch.int32, device=dev),
                 last_action=torch.empty(N, self.act_dim, device=dev), desired_velocity=torch.empty(N, 3, device=dev),
                 fresh=torch.empty(N, dtype=torch.uint8, device=dev))
        _lib.check(self.L.odg_get_env_state(self._h, *[_ptr(o[k]) for k in (
            "step", "gait_index", "gait_matches", "last_action", "desired_velocity", "fresh")], self._stream()),
            "odg_get_env_state")
        return o

    def set_env_state(self, step=None, gait_index=None, gait_matches=None, last_action=None, desired_velocity=None,
                      fresh=None):
        def f(t, dt):
            return None if t is None else torch.as_tensor(t).to(device=self.device, dtype=dt).contiguous()
        args = [f(step, torch.int32), f(gait_index, torch.int32), f(gait_matches, torch.int32),
                f(last_action, torch.float32), f(desired_velocity, torch.float32), f(fresh, torch.uint8)]
        _lib.check(self.L.odg_set_env_state(self._h, *[_ptr(a) for a in args], self._stream()), "odg_set_env_state")
        torch.cuda.current_stream(self.device).synchronize()
