"""Drop-in environment objects with the reference's own surfaces, backed by the batched CUDA simulator.

* `BatchedQuadrupedEnv`  — `QuadrupedEnv` of sim2real/train.py:151-411 for `num_envs` environments on CUDA tensors.
* `QuadrupedEnv`         — the same class name / constructor / numpy 4-tuple API for ONE environment, so
                           `sim2real/train.py` (and its JSON exporter, :600-636) runs unmodified with
                           `from opendog_b200.compat import QuadrupedEnv`.
* `WalkVecEnv`           — `ScaleActionWrapper(WalkEnvironmentV0)` behind the stable-baselines3 `VecEnv` protocol
                           that `train/train.py:63-87,117-130` consumes (numpy in / numpy out, list of info dicts,
                           auto-reset with `terminal_observation`), replacing `SubprocVecEnv`.
Everything computes on the GPU; without the CUDA library or a device these raise (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import lib as _lib
from .env import BatchedWalkEnv, _ptr

REASONS = ("max_steps", "mj_error", "orientation_limit", "too_much_backward")        # sim2real/train.py:393-402
ACTUATOR_NAMES_ORDERED = ["FR_tigh_actuator", "FR_knee_actuator", "FL_tigh_actuator", "FL_knee_actuator",
                          "BR_tigh_actuator", "BR_knee_actuator", "BL_tigh_actuator", "BL_knee_actuator"]


VARIANTS = {"train": 0, "terrain": 1}          # OdgS2RVariant: sim2real/train.py / sim2real/train2.py


class BatchedQuadrupedEnv:
    """`QuadrupedEnv` for `num_envs` environments. variant "train" = sim2real/train.py:151-411 (4 actions, obs 22,
    50 substeps per policy step); variant "terrain" = sim2real/train2.py:159-411 (8 actions, obs 12, 40 substeps)."""

    def __init__(self, num_envs: int, model: str = "our_robot", device=None, auto_reset: bool = True, max_steps: int | None = None,
                 variant: str = "train", first_env_id: int = 0, **sim_config):
        v = VARIANTS[variant]
        # POLICY_DECISION_DT / timestep: 0.10 / 0.002 = 50 mj_step per policy step (train.py:156), 0.08 / 0.002 = 40 (train2.py:106,178)
        # first_env_id: global id of environment 0, so that the random streams of a shard are those of the whole batch
        self.sim = BatchedWalkEnv(num_envs, model=model, device=device, info_keys=None, frame_skip=(50, 40)[v], scale_actions=0,
                                  auto_reset=0, first_env_id=first_env_id, **sim_config)
        self.L, self.device, self.num_envs = self.sim.L, self.sim.device, self.sim.num_envs
        self.first_env_id = int(first_env_id)
        self.variant = variant
        cfg = _lib.OdgS2RConfig()
        self.L.odg_s2r_default_config_for(C.byref(cfg), v)
        cfg.auto_reset = 1 if auto_reset else 0
        self._auto_reset = bool(auto_reset)
        if max_steps is not None:          # MAX_STEPS_PER_EPISODE: 250 (train.py:68) / 1000 (train2.py:88); enforced only with auto_reset
            cfg.max_steps = int(max_steps)
        h = C.c_void_p()
        _lib.check(self.L.odg_s2r_create(self.sim._h, C.byref(self.sim._model), C.byref(cfg), C.byref(h)), "odg_s2r_create")
        self._h = h
        self.state_dim, self.action_dim = self.L.odg_s2r_obs_dim(h), self.L.odg_s2r_act_dim(h)     # 22 / 4 (train.py:164), 12 / 8 (train2.py:186)
        self.obs_dim, self.act_dim = self.state_dim, self.action_dim          # the names opendog_b200.rollout.Rollout reads
        N, dev = num_envs, self.device
        self.obs = torch.empty(N, self.state_dim, device=dev)
        self.reward = torch.empty(N, device=dev)
        self.done = torch.empty(N, dtype=torch.uint8, device=dev)
        self.reason = torch.empty(N, dtype=torch.uint8, device=dev)
        self.sim_target_rad = torch.empty(N, 8, device=dev)
        self.terminal_obs = torch.empty(N, self.state_dim, device=dev)

    def close(self):
        if getattr(self, "_h", None):
            self.L.odg_s2r_destroy(self._h)
            self._h = None
        self.sim.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return self.sim._stream()

    def reset(self, mask=None):
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.L.odg_s2r_reset(self._h, _ptr(m), _ptr(self.obs), self._stream()), "odg_s2r_reset")
        return self.obs

    def _action(self, action):
        a = action
        if a.device != self.device or a.dtype != torch.float32 or not a.is_contiguous():
            a = a.to(device=self.device, dtype=torch.float32).contiguous()
        if a.shape != (self.num_envs, self.action_dim):
            raise ValueError(f"action must be [{self.num_envs}, {self.action_dim}]")
        return a

    def step(self, action: torch.Tensor):
        a = self._action(action)
        _lib.check(self.L.odg_s2r_step(self._h, _ptr(a), _ptr(self.obs), _ptr(self.reward), _ptr(self.done), _ptr(self.reason),
                                       _ptr(self.sim_target_rad), _ptr(self.terminal_obs), self._stream()), "odg_s2r_step")
        info = {"sim_target_rad": self.sim_target_rad, "termination_reason": self.reason, "terminal_obs": self.terminal_obs}
        return self.obs, self.reward, self.done.bool(), info

    def step_into(self, action: torch.Tensor, obs, reward, terminated, truncated):
        """`step` writing obs / reward straight into caller-owned CUDA tensors (rollout buffers), with the episode ends split
        the way `BatchedWalkEnv.step_into` reports them: terminated [N] u8 = a termination condition (reason != RUNNING),
        truncated [N] u8 = the max_steps cap (done with reason RUNNING). `done` and `reason` stay readable on the env.
        No host synchronisation and no allocation: the call can be captured in a CUDA graph."""
        a = self._action(action)
        _lib.check(self.L.odg_s2r_step(self._h, _ptr(a), _ptr(obs), _ptr(reward), _ptr(self.done), _ptr(self.reason),
                                       None, None, self._stream()), "odg_s2r_step")
        # a reason other than RUNNING (0) only comes with done = 1, so terminated = min(reason, 1), truncated = done - terminated
        torch.clamp(self.reason, max=1, out=terminated)
        torch.sub(self.done, terminated, out=truncated)

    def set_bookkeeping(self, counter=None, prev_x=None, cum_pos=None, cum_neg=None, prev_net=None, last_cmd=None):
        def f(t, dt):
            return None if t is None else torch.as_tensor(t).to(device=self.device, dtype=dt).contiguous()
        args = [f(counter, torch.int32), f(prev_x, torch.float64), f(cum_pos, torch.float64), f(cum_neg, torch.float64),
                f(prev_net, torch.float64), f(last_cmd, torch.float32)]
        _lib.check(self.L.odg_s2r_set_bookkeeping(self._h, *[_ptr(a) for a in args], self._stream()), "odg_s2r_set_bookkeeping")
        torch.cuda.current_stream(self.device).synchronize()


class BatchedTerrainQuadrupedEnv(BatchedQuadrupedEnv):
    """The terrain trainer's environment (sim2real/train2.py) with its per-episode height fields: every reset — explicit,
    or the auto-reset of a finished episode — draws a new 100 x 100 terrain for that environment (`TERRAIN_GENERATION_EPISODIC`,
    train2.py:108,307). As in the reference (which loads walking_scene.xml, whose hfield has no geom) the terrain is data
    next to the physics, not part of it: `hfield_data` / `terrain_height` expose it."""

    def __init__(self, num_envs: int, seed: int = 0, first_env_id: int = 0, **kw):
        super().__init__(num_envs, variant="terrain", first_env_id=first_env_id, **kw)
        t = C.c_void_p()
        _lib.check(self.L.odg_terrain_create(num_envs, self.device.index, C.c_uint64(seed), self.first_env_id, C.byref(t)),
                   "odg_terrain_create")
        self._t = t
        self._fields = None

    def close(self):
        if getattr(self, "_t", None):
            self.L.odg_terrain_destroy(self._t)
            self._t = None
        super().close()

    def reset(self, mask=None):
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.L.odg_terrain_generate(self._t, _ptr(m), self._stream()), "odg_terrain_generate")
        return super().reset(mask)

    def _regenerate_done(self):
        if self._auto_reset:
            _lib.check(self.L.odg_terrain_generate(self._t, _ptr(self.done), self._stream()), "odg_terrain_generate")

    def step(self, action):
        out = super().step(action)
        self._regenerate_done()
        return out

    def step_into(self, action, obs, reward, terminated, truncated):
        """As `BatchedQuadrupedEnv.step_into`; the environments that were auto-reset get a new field in the same call (so
        inside a captured CUDA graph too)."""
        super().step_into(action, obs, reward, terminated, truncated)
        self._regenerate_done()

    @property
    def hfield_data(self) -> torch.Tensor:
        """[N, ncol * nrow] float32 view of the device fields, MuJoCo's `model.hfield_data` layout per environment."""
        if self._fields is None:
            iface = {"shape": (self.num_envs, 10000), "typestr": "<f4", "data": (int(self.L.odg_terrain_data(self._t)), False),
                     "version": 3, "strides": None}
            self._fields = torch.as_tensor(type("_Fields", (), {"__cuda_array_interface__": iface})(), device=self.device)
        return self._fields

    def terrain_height(self, xy: torch.Tensor) -> torch.Tensor:
        """`get_terrain_height(x, y)` (train2.py:295-304) for one point per environment: xy [N, 2] -> [N]."""
        q = xy.to(device=self.device, dtype=torch.float32).contiguous()
        h = torch.empty(self.num_envs, device=self.device)
        _lib.check(self.L.odg_terrain_height(self._t, _ptr(q), _ptr(h), self._stream()), "odg_terrain_height")
        return h

    def terrain_from_raw(self, raw: torch.Tensor, radius: torch.Tensor):
        """Test hook: only the deterministic tail of the generator (blend, normalise, transpose) on given raw heights."""
        r = raw.to(device=self.device, dtype=torch.float32).contiguous(); rad = radius.to(device=self.device, dtype=torch.float32).contiguous()
        _lib.check(self.L.odg_terrain_from_raw(self._t, _ptr(r), _ptr(rad), self._stream()), "odg_terrain_from_raw")
        return self.hfield_data


class _DataView:
    """`env.data.qpos / qvel / ctrl` as numpy (fetched from the device on access)."""

    def __init__(self, env):
        self._e = env

    @property
    def qpos(self):
        return self._e._b.sim.get_state()[0][0].double().cpu().numpy()

    @property
    def qvel(self):
        return self._e._b.sim.get_state()[1][0].double().cpu().numpy()

    @property
    def ctrl(self):
        return self._e._b.sim_target_rad[0].double().cpu().numpy()


class QuadrupedEnv:
    """Single-environment numpy façade with the reference's constructor and 4-tuple API (sim2real/train.py:151)."""

    _batched = BatchedQuadrupedEnv
    sim_steps_per_policy_step = 50

    def __init__(self, model_path: str = "our_robot/walking_scene.xml"):
        if "walking_scene" not in str(model_path) and "our_robot" not in str(model_path):
            raise ValueError("QuadrupedEnv supports the OpenDOG walking scene")
        self._b = self._batched(1, auto_reset=False)
        self.state_dim, self.action_dim = self._b.state_dim, self._b.action_dim
        self.viewer = None
        self.model = self._b.sim.desc
        self.data = _DataView(self)
        self.episode_policy_step_counter = 0

    def reset(self):
        self.episode_policy_step_counter = 0
        return self._b.reset()[0].cpu().numpy().astype(np.float32)

    reset_to_home_keyframe = reset

    def step(self, policy_actions_scaled_neg1_to_1):
        a = torch.as_tensor(np.asarray(policy_actions_scaled_neg1_to_1, dtype=np.float32).reshape(1, self.action_dim))
        obs, rew, done, info = self._b.step(a)
        self.episode_policy_step_counter += 1
        reason = int(self._b.reason[0])
        out = {"sim_target_rad": self._b.sim_target_rad[0].double().cpu().numpy(), "termination_reason": REASONS[reason]}
        if reason == 1:
            out["mj_error"] = True
        return obs[0].cpu().numpy().astype(np.float32), float(rew[0]), bool(done[0]), out

    # viewer hooks of the reference are no-ops here
    def launch_viewer_internal(self): return False
    def close_viewer_internal(self): pass
    def sync_viewer_if_active(self): pass
    def close(self): self._b.close()


class TerrainQuadrupedEnv(QuadrupedEnv):
    """Single-environment numpy façade of the terrain trainer's `QuadrupedEnv` (sim2real/train2.py:159-411): 12-float
    observation, 8 actions, the same 4-tuple API; `get_terrain_height(x, y)` and `hfield_data` as the reference exposes them."""
    _batched = BatchedTerrainQuadrupedEnv
    sim_steps_per_policy_step = 40

    @property
    def current_episode_steps(self):
        return self.episode_policy_step_counter

    def get_terrain_height(self, world_x, world_y):
        return float(self._b.terrain_height(torch.tensor([[world_x, world_y]], dtype=torch.float32))[0])

    @property
    def hfield_data(self):
        return self._b.hfield_data[0].cpu().numpy()


def _gym_box(low, high, shape, dtype):
    """A gymnasium Box when gymnasium is importable (SB3 needs the real thing), else a minimal stand-in."""
    try:
        from gymnasium.spaces import Box
        return Box(low, high, shape, dtype)
    except Exception:
        class _Box:
            def __init__(self, low, high, shape, dtype):
                self.low = np.full(shape, low, dtype); self.high = np.full(shape, high, dtype)
                self.shape, self.dtype = tuple(shape), np.dtype(dtype)

            def sample(self):
                lo = np.where(np.isfinite(self.low), self.low, -1.0); hi = np.where(np.isfinite(self.high), self.high, 1.0)
                return np.random.uniform(lo, hi).astype(self.dtype)

            def contains(self, x):
                x = np.asarray(x)
                return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

            def __repr__(self):
                return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"
        return _Box(low, high, shape, dtype)


class _VecEnvProtocol:
    """The abstract interface of `stable_baselines3.common.vec_env.VecEnv` (SB3 2.x), used as the base class when SB3
    itself is not importable. With SB3 installed `WalkVecEnv` subclasses the real `VecEnv`, which is what
    `PPO(..., env=vec_env)` requires: anything else is wrapped as a single gym env (`_wrap_env` -> `_patch_env`)."""

    def __init__(self, num_envs, observation_space, action_space):
        self.num_envs = num_envs
        self.observation_space, self.action_space = observation_space, action_space
        self.reset_infos = [{} for _ in range(num_envs)]
        self._seeds = [None for _ in range(num_envs)]
        self._options = [{} for _ in range(num_envs)]
        self.render_mode = None

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _get_indices(self, indices):
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return indices

    def seed(self, seed=None):
        if seed is None:
            seed = int(np.random.randint(0, np.iinfo(np.uint32).max, dtype=np.uint32))
        self._seeds = [seed + i for i in range(self.num_envs)]
        return self._seeds

    def set_options(self, options=None):
        options = options or {}
        self._options = [dict(options)] * self.num_envs if isinstance(options, dict) else list(options)

    def _reset_seeds(self):
        self._seeds = [None for _ in range(self.num_envs)]

    def _reset_options(self):
        self._options = [{} for _ in range(self.num_envs)]

    @property
    def unwrapped(self):
        return self

    def getattr_depth_check(self, name, already_found):
        return None


def _vecenv_base():
    try:
        from stable_baselines3.common.vec_env import VecEnv
        return VecEnv
    except Exception:
        return _VecEnvProtocol


class LazyInfo(dict):
    """One environment's `info` dict whose per-step entries (WalkEnvironment.py:65-72) are read from the step's host
    arrays on access instead of being copied into N Python dicts every step. Entries that exist only for some
    environments (`terminal_observation`, `TimeLimit.truncated`, `episode`) are ordinary dict items. Behaves like the
    dict SB3's VecMonitor / callbacks expect: `in`, `[]`, `.get`, `.keys/.items`, `.copy()` (a plain dict), assignment."""
    __slots__ = ("_rows", "_i")
    PAWS = (4, 7, 10, 13)                                                   # paw body ids (reward_calc.py:58-63 order)

    def __init__(self, rows, i):
        super().__init__()
        self._rows, self._i = rows, i

    def _lazy(self, k):
        a = self._rows[k][self._i]
        if k == "paw_contact_forces":
            return {b: a[j].astype(np.float64) for j, b in enumerate(self.PAWS)}
        return float(a)

    def __missing__(self, k):
        if k in self._rows:
            v = self._lazy(k)
            dict.__setitem__(self, k, v)
            return v
        raise KeyError(k)

    def __contains__(self, k):
        return dict.__contains__(self, k) or k in self._rows

    def get(self, k, default=None):
        return self[k] if k in self else default

    def keys(self):
        return list(dict.keys(self)) + [k for k in self._rows if not dict.__contains__(self, k)]

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return len(self.keys())

    def items(self):
        return [(k, self[k]) for k in self.keys()]

    def values(self):
        return [self[k] for k in self.keys()]

    def copy(self):
        return dict(self.items())


class WalkVecEnv(_vecenv_base()):
    """`ScaleActionWrapper(WalkEnvironmentV0)` x num_envs behind the stable-baselines3 `VecEnv` interface, replacing
    `make_vec_env(make_env_fn, n_envs, vec_env_cls=SubprocVecEnv)` of train/train.py:63-87. A real `VecEnv` subclass when
    SB3 is importable, so `PPO("MlpPolicy", env=WalkVecEnv(n))` (train/train.py:117-130) takes it as is.

    Per step: one pinned-host action copy in, one fused kernel, ONE device->host copy of the slab holding obs / reward /
    flags / every info array; infos are `LazyInfo` views of that slab. Worker semantics of SB3 (auto-reset on done,
    `terminal_observation`, `TimeLimit.truncated`) come from the kernel; the `Monitor(info_keywords=...)` wrapper each
    reference env gets (train/train.py:69-70) is reproduced here: `info["episode"] = {"r", "l", "t", **keywords}` when an
    episode ends, which is where SB3's `ep_rew_mean` / `ep_len_mean` come from."""

    metadata = {"render_modes": ["human", "rgb_array", "depth_array"], "render_fps": 50}     # WalkEnvironment.py:28-31
    INFO_KEYS = ("x_position", "y_position", "distance_from_origin", "paw_contact_forces", "patterns_matches",
                 "linear_vel_tracking_reward", "reward_ctrl", "terminal_obs")

    def __init__(self, num_envs: int, device=None, seed: int = 0,
                 monitor_info_keywords=("x_position", "y_position", "distance_from_origin", "paw_contact_forces", "patterns_matches"),
                 **config):
        import time
        self.env = BatchedWalkEnv(num_envs, device=device, seed=seed, auto_reset=1, info_keys=self.INFO_KEYS, **config)
        obs_space = _gym_box(-np.inf, np.inf, (self.env.obs_dim,), np.float64)               # WalkEnvironment.py:46-48
        act_space = _gym_box(-1.0, 1.0, (self.env.act_dim,), np.float32)                     # ScaleActionEnvironment.py:19
        super().__init__(num_envs, obs_space, act_space)
        self.observation_shape, self.action_shape = (self.env.obs_dim,), (self.env.act_dim,)
        self.monitor_info_keywords = tuple(monitor_info_keywords or ())
        self._actions = None
        self._h_act = torch.empty(num_envs, self.env.act_dim, pin_memory=True)
        self._t0 = time.time()
        self._ep_ret = np.zeros(num_envs, np.float64)
        self._ep_len = np.zeros(num_envs, np.int64)
        self.render_mode = "rgb_array"

    # ------------------------------------------------------------------ VecEnv interface
    def reset(self):
        obs = self.env.reset().double().cpu().numpy()
        self._ep_ret[:] = 0; self._ep_len[:] = 0
        self.reset_infos = [{} for _ in range(self.num_envs)]
        if hasattr(self, "_reset_seeds"):
            self._reset_seeds(); self._reset_options()
        return obs

    def step_async(self, actions):
        self._actions = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.num_envs, self.env.act_dim)

    def step_wait(self):
        import time
        self._h_act.copy_(torch.from_numpy(self._actions))
        h_obs, h_rew, h_term, h_trunc, h_info = self.env.step_host(self._h_act, with_info=True)
        obs = h_obs.numpy().astype(np.float64)                       # fresh arrays: SB3 keeps them across steps
        rew = h_rew.numpy().astype(np.float64)
        term = h_term.numpy().astype(bool); trunc = h_trunc.numpy().astype(bool)
        done = term | trunc
        rows = {k: v.numpy().copy() for k, v in h_info.items() if k != "terminal_obs"}
        infos = [LazyInfo(rows, i) for i in range(self.num_envs)]
        self._ep_ret += rew; self._ep_len += 1
        if done.any():
            tobs = h_info["terminal_obs"].numpy()
            now = round(time.time() - self._t0, 6)
            for i in np.flatnonzero(done):
                d = infos[i]
                d["terminal_observation"] = tobs[i].astype(np.float64)
                d["TimeLimit.truncated"] = bool(trunc[i] and not term[i])
                ep = {"r": round(float(self._ep_ret[i]), 6), "l": int(self._ep_len[i]), "t": now}     # Monitor.step
                for k in self.monitor_info_keywords:
                    ep[k] = d[k]
                d["episode"] = ep
            self._ep_ret[done] = 0; self._ep_len[done] = 0
        return obs, rew, done, infos

    def close(self):
        self.env.close()

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False for _ in self._get_indices(indices)]

    def get_attr(self, attr_name, indices=None):
        """Attributes of the per-env objects the reference builds: `render_mode`, `metadata`, spaces; anything else is
        looked up on the batched environment."""
        own = {"render_mode": self.render_mode, "metadata": self.metadata, "observation_space": self.observation_space,
               "action_space": self.action_space, "spec": None}
        v = own[attr_name] if attr_name in own else getattr(self.env, attr_name)
        return [v for _ in self._get_indices(indices)]

    def set_attr(self, attr_name, value, indices=None):
        """Per-env attributes do not exist in a batched simulator: a config field of the whole batch can be set for ALL
        envs at once (indices=None); anything narrower is refused rather than silently ignored."""
        if indices is not None and len(list(self._get_indices(indices))) != self.num_envs:
            raise NotImplementedError("WalkVecEnv.set_attr: attributes are shared by the whole batch")
        if attr_name == "render_mode":
            self.render_mode = value
        else:
            raise AttributeError(f"WalkVecEnv has no settable per-env attribute {attr_name!r}")

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        idx = list(self._get_indices(indices))
        if method_name in ("get_wrapper_attr",) and method_args:
            return self.get_attr(method_args[0], indices)
        if method_name == "render":
            return [None for _ in idx]
        raise NotImplementedError(f"WalkVecEnv.env_method({method_name!r}): the batched simulator has no per-env Python object")

    def get_images(self):
        return [None for _ in range(self.num_envs)]           # no renderer on the GPU path (viewers are out of scope)

    def render(self, mode=None):
        return None
