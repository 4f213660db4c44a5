"""The reference's ActorCritic (sim2real/train.py:132-149) with its rollout-time forward on B200 tensor cores.

`ActorCriticB200` keeps the parameters in the reference's own `state_dict` layout (`actor.{0,2,4}.{weight,bias}`,
`critic.*`, `action_log_std`), so a reference `.pth` loads unchanged and a torch optimiser can update them. The
batched forward used while collecting rollouts (`act`) is one of libodgsim's fused tcgen05 kernels (include/odg_policy.h);
`evaluate` — the differentiable forward the PPO/A2C update needs — stays plain torch autograd, as in the reference.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn as nn

from . import lib as _lib


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class ActorCriticB200(nn.Module):
    """`hidden` = the two hidden widths. (512, 256) is sim2real/train.py:135-149 and the benchmark policy; (1024, 512) is
    the terrain trainer's network (sim2real/train2.py:151-153). For both, the rollout-time forward (`act`) is one fused
    tcgen05 kernel launch with the sampling in its epilogue (include/odg_policy.h): the noise is Philox keyed by
    (seed, global row id, step), so sharded and graphed rollouts draw the same noise, and the hidden layers use the
    hardware tanh the update phase's `linear_tanh` uses. Other widths (the reference's older 22-256-256-4 checkpoints) run
    `_act_library`: the same arithmetic as library GEMMs through torch, with noise from a torch generator."""

    def __init__(self, state_dim: int, action_dim: int, action_std_init: float = 0.4, device=None, seed: int = 0,
                 hidden=(512, 256)):
        super().__init__()
        if not torch.cuda.is_available():
            raise _lib.OdgError("ActorCriticB200 needs a CUDA device: opendog_b200 has no CPU fallback")
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.dev.index is None:
            self.dev = torch.device("cuda", torch.cuda.current_device())
        self.state_dim, self.action_dim, self.seed = state_dim, action_dim, seed
        h1, h2 = int(hidden[0]), int(hidden[1])
        self.hidden = (h1, h2)
        self.fused = self.hidden in ((512, 256), (1024, 512))          # the widths libodgsim's forward kernels cover
        self.actor = nn.Sequential(nn.Linear(state_dim, h1), nn.Tanh(), nn.Linear(h1, h2), nn.Tanh(),
                                   nn.Linear(h2, action_dim), nn.Tanh())
        self.critic = nn.Sequential(nn.Linear(state_dim, h1), nn.Tanh(), nn.Linear(h1, h2), nn.Tanh(),
                                    nn.Linear(h2, 1))
        self.action_log_std = nn.Parameter(torch.ones(1, action_dim) * math.log(action_std_init))
        self.to(self.dev)
        self.L = _lib.load()
        self._h = None
        self._launches = 0
        self._gen = torch.Generator(device=self.dev)
        self._gen.manual_seed(seed)
        if self.fused:
            h = C.c_void_p()
            _lib.check(self.L.odg_policy_create_hidden(state_dim, action_dim, h1, h2, self.dev.index, C.byref(h)),
                       "odg_policy_create_hidden")
            self._h = h
        self._step = 0
        self.sync_weights()

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self.L.odg_policy_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    @property
    def launch_count(self) -> int:
        return int(self.L.odg_policy_launch_count(self._h)) if self.fused else self._launches

    def sync_weights(self):
        """Re-pack the fp32 parameters into the kernel's bf16 operand layout (call after every optimiser step
        or load_state_dict)."""
        if not self.fused:
            return
        w = _lib.OdgPolicyWeights()
        keep = []
        for name, net in (("actor", self.actor), ("critic", self.critic)):
            for i, li in enumerate((0, 2, 4)):
                wt = net[li].weight.detach().contiguous().float()
                bs = net[li].bias.detach().contiguous().float()
                keep += [wt, bs]
                getattr(w, name + "_w")[i] = wt.data_ptr()
                getattr(w, name + "_b")[i] = bs.data_ptr()
        ls = self.action_log_std.detach().reshape(-1).contiguous().float()
        keep.append(ls)
        w.action_log_std = ls.data_ptr()
        _lib.check(self.L.odg_policy_load(self._h, C.byref(w), self._stream()), "odg_policy_load")
        self._pack_keep = keep       # the packing kernels run asynchronously: their fp32 sources stay referenced until the next call

    # ------------------------------------------------------------------ rollout-time forward (tensor cores)
    def act(self, obs: torch.Tensor, sample: bool = True, out=None, first_row_id: int = 0, step: int | None = None,
            step_base: torch.Tensor | None = None):
        """(action, logp, value, mean) for obs [N, state_dim]; `sample=False` returns the mean as the action
        (the reference's export path, sim2real/train.py:613). `out` = dict of preallocated tensors (optional)."""
        o = obs
        if o.device != self.dev or o.dtype != torch.float32 or not o.is_contiguous():
            o = o.to(device=self.dev, dtype=torch.float32).contiguous()
        n = o.shape[0]
        out = out or {}
        if not self.fused:
            return self._act_library(o, sample, out)
        mean = out.get("mean") if out.get("mean") is not None else torch.empty(n, self.action_dim, device=self.dev)
        value = out.get("value") if out.get("value") is not None else torch.empty(n, device=self.dev)
        action = logp = None
        if sample:
            action = out.get("action") if out.get("action") is not None else torch.empty(n, self.action_dim, device=self.dev)
            logp = out.get("logp") if out.get("logp") is not None else torch.empty(n, device=self.dev)
        if step is None:
            step = self._step
            self._step += 1
        _lib.check(self.L.odg_policy_forward(self._h, _ptr(o), n, _ptr(mean), _ptr(value), _ptr(action), _ptr(logp),
                                             C.c_uint64(self.seed), C.c_uint32(step & 0xFFFFFFFF), _ptr(step_base), first_row_id,
                                             self._stream()), "odg_policy_forward")
        return (action if sample else mean), logp, value, mean

    @torch.no_grad()
    def _act_library(self, o, sample, out):
        """Rollout-time forward for hidden sizes neither fused kernel covers: bf16 operands, fp32 accumulation, on the
        device (cuBLAS through torch). The noise comes from a torch generator, not the kernels' keyed Philox stream."""
        with torch.autocast("cuda", dtype=torch.bfloat16):
            mean = self.actor(o).float()
            value = self.critic(o).float().squeeze(-1)
        self._launches += 1
        ls = self.action_log_std.detach().reshape(-1)
        action = logp = None
        if sample:
            eps = torch.randn(mean.shape, device=self.dev, generator=self._gen)
            action = mean + torch.exp(ls) * eps
            logp = (-0.5 * eps * eps - ls - 0.9189385332046727).sum(-1)
        for k, v in (("mean", mean), ("value", value), ("action", action), ("logp", logp)):
            if v is not None and out.get(k) is not None:
                out[k].copy_(v)
        pick = lambda k, v: out[k] if out.get(k) is not None else v
        mean, value = pick("mean", mean), pick("value", value)
        if sample:
            action, logp = pick("action", action), pick("logp", logp)
        return (action if sample else mean), logp, value, mean

    # ------------------------------------------------------------------ differentiable forward (update phase)
    def forward(self, state):
        """Same signature as the reference module: (Normal(mean, std), value)."""
        mean = self.actor(state)
        std = torch.exp(self.action_log_std.expand_as(mean))
        return torch.distributions.Normal(mean, std, validate_args=False), self.critic(state)

    # the update-phase forward on padded inputs: with the observation width rounded up to a multiple of 16 (33 -> 48,
    # zero columns in x and W1) every GEMM of the forward and backward pass is tensor-core aligned in bf16; with K = 33
    # cuBLAS falls back to legacy kernels that take a third of the whole PPO epoch (tools/prof_ppo.py)
    @staticmethod
    def pad_obs(state, multiple: int = 16):
        k = (-state.shape[-1]) % multiple
        return torch.nn.functional.pad(state, (0, k)) if k else state

    def forward_padded(self, state_padded):
        F = torch.nn.functional
        k = state_padded.shape[-1] - self.state_dim
        def run(net):
            x = linear_tanh(state_padded, F.pad(net[0].weight, (0, k)), net[0].bias)
            x = linear_tanh(x, net[2].weight, net[2].bias)
            w3, b3 = net[4].weight, net[4].bias
            n3 = w3.shape[0]
            if n3 % 8 and x.is_cuda:
                # a head narrower than 8 outputs (the critic's single value): zero rows up to 8, so that its backward GEMMs
                # (K = out_features) are tensor-core aligned too — with K = 1 cuBLAS takes a legacy align-1 kernel
                p3 = (-n3) % 8
                return F.linear(x, F.pad(w3, (0, 0, 0, p3)), F.pad(b3, (0, p3)))[:, :n3]
            return F.linear(x, w3, b3)
        mean = torch.tanh(run(self.actor))
        std = torch.exp(self.action_log_std.expand_as(mean))
        # (validate_args=False: the argument check reads a flag back to the host — a device sync per forward, and illegal
        #  inside a CUDA-graph capture)
        return torch.distributions.Normal(mean, std, validate_args=False), run(self.critic)


class _LinearTanh(torch.autograd.Function):
    """`tanh(linear(x, w, b))` of a hidden layer in the update phase, bf16 operands (what autocast makes of it), with a
    backward whose tanh derivative and bias gradient are ONE pass over the activation gradient (include/odg_policy.h:
    odg_tanh_backward_bias) instead of torch's two (tanh_backward, then a bf16 column reduction)."""

    @staticmethod
    def forward(ctx, x, w, b):
        with torch.autocast("cuda", enabled=False):
            xb, wb = x.to(torch.bfloat16), w.to(torch.bfloat16)
            y = torch.nn.functional.linear(xb, wb, b.to(torch.bfloat16))
        if y.is_contiguous() and y.numel() % 8 == 0:
            st = C.c_void_p(torch.cuda.current_stream(y.device).cuda_stream)        # in place, the rollout kernel's tanh
            _lib.check(_lib.load().odg_tanh_bf16(_ptr(y), _ptr(y), y.numel(), st), "odg_tanh_bf16")
        else:
            y = torch.tanh(y)
        ctx.save_for_backward(xb, wb, y)
        ctx.dtypes = (x.dtype, w.dtype, b.dtype)
        return y

    @staticmethod
    def backward(ctx, gy):
        xb, wb, y = ctx.saved_tensors
        L = _lib.load()
        rows, cols = y.shape
        gy = gy.to(torch.bfloat16).contiguous()
        g = torch.empty_like(y)
        gb = torch.empty(cols, device=y.device, dtype=torch.float32)
        scratch = torch.empty(L.odg_tanh_backward_bias_scratch_floats(cols), device=y.device, dtype=torch.float32)
        st = C.c_void_p(torch.cuda.current_stream(y.device).cuda_stream)
        _lib.check(L.odg_tanh_backward_bias(_ptr(gy), _ptr(y), _ptr(g), _ptr(gb), _ptr(scratch), rows, cols, st),
                   "odg_tanh_backward_bias")
        dx, dw, db = ctx.dtypes
        with torch.autocast("cuda", enabled=False):
            gx = (g @ wb).to(dx) if ctx.needs_input_grad[0] else None
            gw = (g.t() @ xb).to(dw) if ctx.needs_input_grad[1] else None
        return gx, gw, (gb.to(db) if ctx.needs_input_grad[2] else None)


def linear_tanh(x, w, b):
    """Hidden layer of the update-phase forward: the fused-backward form on CUDA under bf16 autocast when the width allows
    it (8 x a power of two, every ActorCritic of the reference: 512 / 256, 1024 / 512), plain torch otherwise (the TF32
    path without autocast; CPU runs of the gloo tests)."""
    n = w.shape[0]
    if (x.is_cuda and torch.is_autocast_enabled() and x.dim() == 2 and n % 8 == 0 and n <= 2048
            and ((n // 8) & (n // 8 - 1)) == 0):
        return _LinearTanh.apply(x, w, b)
    return torch.tanh(torch.nn.functional.linear(x, w, b))


class _PPOLoss(torch.autograd.Function):
    """Clipped-surrogate loss of one minibatch with its gradients computed in the same pass (include/odg_policy.h:
    odg_ppo_loss). Returns (loss, terms) with terms = [loss, pg, vf, entropy] (not differentiable)."""

    @staticmethod
    def forward(ctx, mean, value, log_std, action, logp_old, adv, ret, clip, vf_coef, ent_coef):
        L = _lib.load()
        dev = mean.device
        B, A = mean.shape
        f = lambda t: t.detach().to(torch.float32).contiguous()
        m, v, ls = f(mean), f(value).reshape(-1), f(log_std).reshape(-1)
        loss = torch.empty((), device=dev); terms = torch.empty(4, device=dev)
        g_mean = torch.empty(B, A, device=dev); g_value = torch.empty(B, device=dev); g_ls = torch.empty(A, device=dev)
        scratch = torch.empty(L.odg_ppo_loss_scratch_floats(), device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(L.odg_ppo_loss(_ptr(m), _ptr(v), _ptr(ls), _ptr(f(action)), _ptr(f(logp_old)), _ptr(f(adv)), _ptr(f(ret)),
                                  B, A, float(clip), float(vf_coef), float(ent_coef), _ptr(loss), _ptr(terms), _ptr(g_mean),
                                  _ptr(g_value), _ptr(g_ls), _ptr(scratch), st), "odg_ppo_loss")
        ctx.save_for_backward(g_mean, g_value, g_ls)
        ctx.meta = (mean.dtype, value.dtype, value.shape, log_std.dtype, log_std.shape)
        ctx.mark_non_differentiable(terms)
        return loss, terms

    @staticmethod
    def backward(ctx, gl, _gterms):
        g_mean, g_value, g_ls = ctx.saved_tensors
        md, vd, vs, ld, lshape = ctx.meta
        return ((g_mean * gl).to(md), (g_value * gl).reshape(vs).to(vd), (g_ls * gl).reshape(lshape).to(ld),
                None, None, None, None, None, None, None)


def ppo_loss(mean, value, log_std, action, logp_old, adv, ret, clip, vf_coef, ent_coef):
    """(loss, pg, vf, entropy) of the clipped-surrogate objective for a diagonal Normal(mean, exp(log_std)) policy: one fused
    kernel on CUDA (forward and gradients), the plain torch expression elsewhere (CPU runs of the gloo tests; wider actions)."""
    if mean.is_cuda and mean.dim() == 2 and mean.shape[1] <= 16:
        loss, terms = _PPOLoss.apply(mean, value, log_std, action, logp_old, adv, ret, clip, vf_coef, ent_coef)
        return loss, terms[1], terms[2], terms[3]
    d = torch.distributions.Normal(mean, torch.exp(log_std.expand_as(mean)), validate_args=False)
    logp = d.log_prob(action).float().sum(-1)
    ratio = torch.exp(logp - logp_old)
    pg = -torch.min(ratio * adv, torch.clamp(ratio, 1 - clip, 1 + clip) * adv).mean()
    vf = torch.nn.functional.mse_loss(value.float().reshape(-1), ret)
    ent = d.entropy().float().sum(-1).mean()
    return pg + vf_coef * vf - ent_coef * ent, pg, vf, ent


def gae(reward, value, done, gamma=0.99, lam=0.95, normalize=True, group=None):
    """GAE + advantage normalisation (sim2real/train.py:557-564) for [T, N] rollouts on the GPU.

    reward [T,N] f32, value [T+1,N] f32 (last row = bootstrap), done [T,N] bool/uint8. With `group` (a
    torch.distributed process group, NCCL) the advantage statistics [sum, sumsq, count] are all-reduced so
    every rank normalises with the statistics of the whole job. Returns (adv, returns, stats)."""
    L = _lib.load()
    T, N = reward.shape
    dev = reward.device
    reward = reward.contiguous().float()
    value = value.contiguous().float()
    done = done.contiguous().to(torch.uint8)
    adv = torch.empty(T, N, device=dev)
    ret = torch.empty(T, N, device=dev)
    stats = torch.empty(3, dtype=torch.float64, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(L.odg_gae(_ptr(reward), _ptr(value), _ptr(done), T, N, gamma, lam, _ptr(adv), _ptr(ret), _ptr(stats), st),
               "odg_gae")
    from .train import allreduce_advantage_stats
    allreduce_advantage_stats(stats, group)          # group=False: never; None / True: the default group when initialised
    if normalize:
        count = int(T * N)
        _lib.check(L.odg_normalize_advantages(_ptr(adv), count, _ptr(stats), st), "odg_normalize_advantages")
    return adv, ret, stats
