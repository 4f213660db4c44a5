"""GPU tests of the rollout kernels (through the C ABI): tcgen05 policy MLP vs a torch reference of the same
ActorCritic (sim2real/train.py:132-149), sampling / log-prob vs a numpy restatement of the Philox stream, GAE vs
the reference's Python loop (sim2real/train.py:557-564); and the PPO update-phase kernels (odg_tanh_bf16,
odg_tanh_backward_bias, odg_ppo_loss) vs float64 references, up to the configs[3] minibatch of 393216 rows where their
grid-stride and unrolled loops run. Outputs are guard-banded: written past their end, a sentinel tail changes.

Tolerances of the policy forward: the kernel computes with bf16 operands and fp32 accumulation. Against a torch model that rounds inputs,
weights and hidden activations to bf16 the outputs agree to 4e-3 (tanh.approx + accumulation order); against the
plain fp32 torch model to 3e-2 (bf16 quantisation of a 512-wide layer)."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu


def _bf16(x):
    return x.to(torch.bfloat16).to(torch.float32)


# ---- guard bands: an output is the head of a larger buffer whose every element starts as a NaN payload no kernel writes;
# the tail must still hold it after the call (a masked store or a grid-stride tail that runs one element too far fails)
_SENTINEL = {torch.float32: (torch.int32, 0x7FA1B2C3), torch.bfloat16: (torch.int16, 0x7FB5)}


class _Guarded:
    def __init__(self, shape, dtype=torch.float32, tail=256):
        self.n = math.prod(shape)
        self.buf = torch.empty(self.n + tail, dtype=dtype, device="cuda")
        ityp, bits = _SENTINEL[dtype]
        self.buf.view(ityp).fill_(bits)
        self.t = self.buf[:self.n].view(shape)

    def assert_tail_intact(self, what):
        ityp, bits = _SENTINEL[self.buf.dtype]
        bad = int((self.buf.view(ityp)[self.n:] != bits).sum())
        assert bad == 0, f"{what}: {bad} elements written past the end of the output"


def _cptr(t):
    import ctypes as C
    return C.c_void_p(t.data_ptr())


def _stream():
    import ctypes as C
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _pow2(k):
    """2.0 ** k, exactly, for an integer tensor k in the normal float64 range (built from the exponent bits)."""
    return ((k.to(torch.int64) + 1023) << 52).view(torch.float64)


def _bf16_rn(x64):
    """(the correctly rounded (nearest, ties to even) bf16 value of float64 `x64`, as float64; the relative distance of
    x64 from the nearest bf16 rounding midpoint). Normal bf16 range."""
    m, e = torch.frexp(x64)
    f = m * 256.0                                        # |f| in [128, 256): the 8 significant bits, the rest a fraction
    a = f.abs()
    return torch.round(f) * _pow2(e - 8), ((a - a.floor()) - 0.5).abs() / a.clamp_min(1.0)


def _philox_np(seed, c0, c1, c2, c3):
    """Philox4x32-10 (odg_core.cuh: philox4x32) on numpy uint32 counter arrays: the four output words."""
    c = [np.asarray(x, dtype=np.uint64) & 0xFFFFFFFF for x in (c0, c1, c2, c3)]
    c = [x.astype(np.uint64) for x in np.broadcast_arrays(*c)]
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & m32]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return [x.astype(np.uint32) for x in c]


def _sample_eps_np(seed, rows, step, A):
    """The policy kernel's Normal noise for global row ids `rows`: eps [len(rows), A] in float64 from Philox4x32-10 keyed by
    (seed, row, step, block of 4 action dims, stream "SAMP"), two Box-Muller pairs per block (odg_policy.cu: sample_actor)."""
    eps = []
    for blk in range((A + 3) // 4):
        r = _philox_np(seed, rows, step, blk, 0x53414D50)
        for pr in range(2):
            u1 = ((r[2 * pr] >> 8).astype(np.float64) + 1.0) * 2.0 ** -24          # (0, 1]
            u2 = (r[2 * pr + 1] >> 8).astype(np.float64) * 2.0 ** -24              # [0, 1)
            rad = np.sqrt(-2.0 * np.log(u1))
            eps += [rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)]
    return np.stack(eps[:A], axis=1)


def test_vectorised_philox_matches_the_oracle():
    """The numpy Philox restatement the sampling checks use against the oracle's C philox4x32 (CPU only)."""
    from oracle.oracle import philox
    rng = np.random.default_rng(3)
    n = 300
    cs = [rng.integers(0, 2 ** 32, n, dtype=np.uint64) for _ in range(4)]
    cs[0][:3] = [0, 0xFFFFFFFF, 7 * 65536]
    for seed in (7, 0x299F31D0A4093822):
        out = _philox_np(seed, *cs)
        for i in range(n):
            assert [int(o[i]) for o in out] == philox(seed, *(int(c[i]) for c in cs)), (seed, i)


def _ref_forward(m, obs, emulate_bf16):
    def run(net, x, last_tanh):
        for li in (0, 2, 4):
            w, b = net[li].weight.detach(), net[li].bias.detach()
            if emulate_bf16:
                x = _bf16(x) @ _bf16(w).T + b
            else:
                x = x @ w.T + b
            if li != 4 or last_tanh:
                x = torch.tanh(x)
        return x
    return run(m.actor, obs, True), run(m.critic, obs, False)[:, 0]


# (S, A, N, first_row_id). N = "W" is about one full wave of the kernel (1 CTA of 128 rows per SM); cluster placement
# may leave SMs idle, so W + 1 and 65536 / 65537 (3.5 waves at configs[3]'s 65536 environments per GPU) are what make
# CTAs follow others on the same SM (TMEM alloc / dealloc, mbarrier init). first_row_id 7 * 65536 is rank 7's. The
# (S, A) edges exercise K padding (S = 1, 17, 63) and partial Box-Muller blocks (A = 1, 3, 5).
_MLP_CASES = [pytest.param(S, A, N, 1000, id=f"{S}-{A}-{N}") for S, A, N in ((33, 8, 300), (22, 4, 128), (48, 12, 1000), (64, 16, 129))]
_MLP_CASES += [(33, 8, n, 7 * 65536) for n in (16384, "W", "W+1", 65536, 65537)]
_MLP_CASES += [(S, A, 2049, 7 * 65536) for S in (1, 16, 17, 63) for A in (1, 3, 5)]


@gpu
@pytest.mark.parametrize("S,A,N,first_row", _MLP_CASES)
def test_policy_mlp_matches_torch(S, A, N, first_row):
    """`k_mlp` against the torch model for every row (mean, value), and its sampling against the numpy restatement of the
    Philox / Box-Muller stream for every row (action, logp). Every output is guard-banded by at least one CTA's 128 rows,
    so a store by a row past N lands in the sentinel tail."""
    from opendog_b200.policy import ActorCriticB200
    if isinstance(N, str):
        W = 128 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        N = W + (1 if N == "W+1" else 0)
    torch.manual_seed(S * 100 + A)
    m = ActorCriticB200(S, A, 0.4, seed=7)
    with torch.no_grad():
        for p in m.parameters():
            if p.dim() == 2 and p.shape[0] > 16:
                p.mul_(2.0)                      # push hidden units into the non-linear range of tanh
        m.action_log_std.copy_(torch.linspace(-1.5, -0.5, A)[None])
    m.sync_weights()
    obs = torch.randn(N, S, device="cuda") * 1.5
    out = {"mean": _Guarded((N, A), tail=128 * A), "action": _Guarded((N, A), tail=128 * A),
           "value": _Guarded((N,)), "logp": _Guarded((N,))}
    action, logp, value, mean = m.act(obs, step=3, first_row_id=first_row, out={k: g.t for k, g in out.items()})
    torch.cuda.synchronize()
    for k, g in out.items():
        g.assert_tail_intact(k)
    assert mean.data_ptr() == out["mean"].t.data_ptr() and logp.data_ptr() == out["logp"].t.data_ptr()
    r_mean, r_val = _ref_forward(m, obs, True)
    assert (mean - r_mean).abs().max().item() < 4e-3
    assert (value - r_val).abs().max().item() < 4e-3 * max(1.0, r_val.abs().max().item())
    f_mean, f_val = _ref_forward(m, obs, False)
    assert (mean - f_mean).abs().max().item() < 3e-2
    assert (value - f_val).abs().max().item() < 3e-2 * max(1.0, f_val.abs().max().item())
    # sampling, every row: action = mean + exp(log_std) * eps with eps from Philox (seed, first_row + row, step, block)
    ls = m.action_log_std.detach().cpu().double().numpy().reshape(-1)
    act = action.cpu().double().numpy(); mu = mean.cpu().double().numpy(); lp = logp.cpu().double().numpy()
    eps = _sample_eps_np(7, first_row + np.arange(N, dtype=np.uint64), 3, A)
    assert np.abs(act - (mu + np.exp(ls) * eps)).max() < 1e-4
    assert np.abs(lp - np.sum(-0.5 * eps ** 2 - ls - 0.5 * math.log(2 * math.pi), axis=1)).max() < 1e-3
    # the eps of a whole batch look standard normal
    z = ((action - mean) / torch.exp(m.action_log_std)).flatten()
    assert abs(z.mean().item()) < 0.15 and abs(z.std().item() - 1.0) < 0.15
    # deterministic path
    a2, lp2, v2, mean2 = m.act(obs, sample=False)
    assert lp2 is None and torch.equal(a2, mean2) and torch.equal(mean2, mean)


@gpu
def test_gae_matches_reference_loop():
    _check_gae(24, 777)


@gpu
@pytest.mark.parametrize("T,N", [(24, 65536), (3, 257), (1, 3)])
def test_gae_matches_reference_loop_at_more_shapes(T, N):
    """configs[3]'s 24 x 65536 and ragged sizes. (T * N = 1 is left out: torch's std of one element is NaN, where
    odg_normalize_advantages returns 0.)"""
    _check_gae(T, N)


def _check_gae(T, N):
    """`odg_gae` against the reference's loop in float64 for a [T, N] rollout with episodes that end on the last step and
    environments that are done at every step; adv and ret guard-banded; then the normalised advantages."""
    from opendog_b200 import lib as _lib
    from opendog_b200.policy import gae
    L = _lib.load()
    g = torch.Generator().manual_seed(T * N)
    rew = torch.randn(T, N, generator=g); val = torch.randn(T + 1, N, generator=g)
    done = torch.rand(T, N, generator=g) < 0.1
    done[T - 1, ::5] = True                          # episodes that end on the last collected step
    done[:, ::13] = True                             # environments done at every step
    rew_d, val_d, done_d = rew.cuda(), val.cuda(), done.to(torch.uint8).cuda()
    adv_g, ret_g = _Guarded((T, N)), _Guarded((T, N))
    stats = torch.empty(3, dtype=torch.float64, device="cuda")
    _lib.check(L.odg_gae(_cptr(rew_d), _cptr(val_d), _cptr(done_d), T, N, 0.99, 0.95, _cptr(adv_g.t), _cptr(ret_g.t),
                         _cptr(stats), _stream()), "odg_gae")
    torch.cuda.synchronize()
    adv_g.assert_tail_intact("adv"); ret_g.assert_tail_intact("ret")
    adv, ret = adv_g.t, ret_g.t
    # sim2real/train.py:557-561 per environment
    r64, v64, m64 = rew.double().numpy(), val.double().numpy(), (~done).double().numpy()
    ref = np.zeros((T, N)); a = np.zeros(N)
    for t in reversed(range(T)):
        delta = r64[t] + 0.99 * v64[t + 1] * m64[t] - v64[t]
        a = delta + 0.99 * 0.95 * m64[t] * a
        ref[t] = a
    assert np.abs(adv.cpu().numpy() - ref).max() < 1e-4
    assert np.abs(ret.cpu().numpy() - (ref + v64[:T])).max() < 1e-4
    s = stats.cpu().numpy()
    a32 = adv.cpu().double().numpy()
    assert abs(s[0] - a32.sum()) < 1e-6 * max(1, abs(a32.sum())) + 1e-6 and abs(s[1] - (a32 ** 2).sum()) < 1e-6 * (a32 ** 2).sum()
    assert s[2] == T * N
    adv_n, _, _ = gae(rew.cuda(), val.cuda(), done.cuda(), 0.99, 0.95, normalize=True, group=False)
    ref_n = (torch.from_numpy(ref).float() - torch.from_numpy(ref).float().mean()) / (torch.from_numpy(ref).float().std() + 1e-8)
    assert (adv_n.cpu() - ref_n).abs().max().item() < 1e-4


@gpu
def test_rollout_graph_equals_eager_and_feeds_gae():
    """One horizon collected through the CUDA graph equals the same horizon collected launch by launch."""
    from opendog_b200.env import BatchedWalkEnv
    from opendog_b200.policy import ActorCriticB200
    from opendog_b200.rollout import Rollout
    outs = []
    for use_graph in (False, True):
        torch.manual_seed(0)
        env = BatchedWalkEnv(96, seed=5, info_keys=None, max_episode_steps=30)
        pol = ActorCriticB200(env.obs_dim, env.act_dim, 0.4, seed=11)
        ro = Rollout(env, pol, horizon=12, use_graph=use_graph)
        for _ in range(3):                       # the graph path warms up once, captures once, then replays
            ro.collect()
        torch.cuda.synchronize()
        outs.append([x.clone() for x in (ro.obs, ro.action, ro.logp, ro.value, ro.reward, ro.done)])
        adv, ret, stats = ro.advantages(normalize=True, group=False)
        assert torch.isfinite(adv).all() and abs(adv.mean().item()) < 1e-3 and abs(adv.std().item() - 1) < 1e-3
    # the eager run did 3 collects; the graph run did warm-up + capture + 1 replay = 3 collects as well
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert outs[0][5].any(), "episodes should end (truncation at 30) inside the last collected horizon (steps 25-36)"


@gpu
@pytest.mark.parametrize("use_graph", [False, True])
def test_first_horizon_starts_from_the_reset_observation(use_graph):
    """ADVICE r1: the first collect() must act on the `env.reset()` observation (not on a zero row), and in every horizon
    it returns — eager, the eager warm-up of the graph path, the capture + first replay, later replays — obs[t] must be the
    observation that action[t] / logp[t] were computed from."""
    from opendog_b200.env import BatchedWalkEnv
    from opendog_b200.policy import ActorCriticB200
    from opendog_b200.rollout import Rollout
    env = BatchedWalkEnv(160, seed=8, info_keys=None)
    pol = ActorCriticB200(env.obs_dim, env.act_dim, 0.4, seed=3)
    ro = Rollout(env, pol, horizon=6, use_graph=use_graph)
    reset_obs = ro.obs[0].clone()
    assert reset_obs.abs().sum().item() > 0
    std = torch.exp(pol.action_log_std.detach()).reshape(-1)
    last = None
    for k in range(4):
        ro.collect()
        torch.cuda.synchronize()
        if k == 0:
            assert torch.equal(ro.obs[0], reset_obs), "row 0 of the first horizon is the reset observation"
        else:
            assert torch.equal(ro.obs[0], last), "row 0 carries the previous horizon's last observation"
        for t in (0, ro.T - 1):
            mean = pol.act(ro.obs[t].clone(), sample=False)[3]
            z = (ro.action[t] - mean) / std
            logp = (-0.5 * z * z - torch.log(std) - 0.5 * math.log(2 * math.pi)).sum(-1)
            assert (logp - ro.logp[t]).abs().max().item() < 2e-3, (k, t)
        last = ro.obs[ro.T].clone()


@gpu
def test_reference_checkpoint_loads_and_runs_through_the_kernel(tmp_path):
    """SURVEY section 5 (checkpoint/resume): a `.pth` written by the reference's own trainer
    (sim2real/train.py:587-588, `torch.save(agent.state_dict())`; fixture = its shipped
    sim2real/output/pth/quadruped_ac_sym_ep3700.pth, 22 -> 512 -> 256 -> 4) loads unchanged into ActorCriticB200, the
    tcgen05 forward reproduces the reference module's torch forward at the stated bf16 tolerances, and the deterministic
    closed-loop rollout + JSON export of sim2real/train.py:600-636 runs on it with the structural invariants of the
    symmetric-trot mapping (train.py:243-259) and the ctrlrange clip (:276)."""
    import json
    import os
    import torch.nn as nn
    from opendog_b200.compat import BatchedQuadrupedEnv
    from opendog_b200.gait import export_walk_json, TRAIN_REAL_HOME_DEG
    from opendog_b200.policy import ActorCriticB200
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_quadruped_ac_sym_ep3700.pth")
    sd = torch.load(path, map_location="cpu", weights_only=True)

    class RefActorCritic(nn.Module):                    # the reference module, restated (sim2real/train.py:132-149)
        def __init__(self, s, a):
            super().__init__()
            self.actor = nn.Sequential(nn.Linear(s, 512), nn.Tanh(), nn.Linear(512, 256), nn.Tanh(), nn.Linear(256, a), nn.Tanh())
            self.critic = nn.Sequential(nn.Linear(s, 512), nn.Tanh(), nn.Linear(512, 256), nn.Tanh(), nn.Linear(256, 1))
            self.action_log_std = nn.Parameter(torch.zeros(1, a))
    ref = RefActorCritic(22, 4)
    ref.load_state_dict(sd)                             # strict: same keys, same shapes
    pol = ActorCriticB200(22, 4, 0.4)
    missing, unexpected = pol.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    pol.sync_weights()
    env = BatchedQuadrupedEnv(256, auto_reset=True)
    obs = env.reset().clone()
    g = torch.Generator(device="cuda").manual_seed(0)
    for t in range(6):                                  # observations the policy actually sees, plus random ones
        x = obs if t % 2 == 0 else torch.randn(256, 22, device="cuda", generator=g)
        mean, _, value, _ = pol.act(x, sample=False)
        with torch.no_grad():
            rm = ref.actor(x.cpu()); rv = ref.critic(x.cpu())[:, 0]
            bm, bv = _ref_forward(ref, x.cpu(), True)
        # (a trained critic's values reach ~20 here, not O(1) as for a fresh network: bf16 rounding errors scale with the
        #  magnitude of the partial sums, so the value tolerances are relative to the batch's largest |value|)
        vs = max(1.0, rv.abs().max().item())
        assert (mean.cpu() - rm).abs().max().item() < 3e-2 and (value.cpu() - rv).abs().max().item() < 3e-2 * vs
        assert (mean.cpu() - bm).abs().max().item() < 4e-3 and (value.cpu() - bv).abs().max().item() < 4e-3 * vs
        obs, _, _, _ = env.step(mean)
        obs = obs.clone()
    out = tmp_path / "walk.json"
    env2 = BatchedQuadrupedEnv(4, auto_reset=False)
    export_walk_json(pol, env2, str(out), num_steps=50)
    steps = json.load(open(out))
    assert len(steps) >= 5 and all(s["duration"] == 0.1 and len(s["targets_deg"]) == 8 for s in steps)
    H = TRAIN_REAL_HOME_DEG
    tol = 0.011                                         # targets are rounded to 2 decimals (train.py:628)
    for k, s in enumerate(steps):
        d = {n: s["targets_deg"][n] - H[n] for n in H}
        # BL mirrors FR and BR mirrors FL on the thighs (train.py:243-247); thigh targets are clipped to ctrlrange
        # [2.36, 2.8] around home 2.35619: delta in [+0.22, +25.43] degrees (our_robot.xml:14-15)
        assert abs(d["BL_tigh_actuator"] - d["FR_tigh_actuator"]) <= tol and abs(d["BR_tigh_actuator"] - d["FL_tigh_actuator"]) <= tol
        for n in ("FR_tigh_actuator", "FL_tigh_actuator"):
            assert 0.21 <= d[n] <= 25.44
        # the stance pair's knees stay home, the swinging pair's knees are antisymmetric (:249-259) up to the ctrlrange clip
        # [-1.8, -1.2] around home -1.5708: delta in [-13.13, +21.25] degrees (our_robot.xml:19-20); phases alternate
        swing, stance = (("FR_knee_actuator", "BL_knee_actuator"), ("FL_knee_actuator", "BR_knee_actuator"))[::1 if k % 2 == 0 else -1]
        assert abs(d[stance[0]]) <= tol and abs(d[stance[1]]) <= tol
        a, b = d[swing[0]], d[swing[1]]
        assert -13.14 <= a <= 21.26 and -13.14 <= b <= 21.26
        clipped = min(a, b) <= -13.12 or max(a, b) >= 21.24
        assert abs(a + b) <= 2 * tol or clipped


@gpu
def test_graphed_ppo_update_equals_the_eager_update():
    """train.GraphedPPOUpdate (the PPO epoch of BASELINE configs[3] replayed as CUDA graphs) against train.ppo_update on
    the same batch from the same initial weights: same losses, same updated parameters (both run the bf16-autocast
    forward / backward; the graph only removes launch and allocator time)."""
    from opendog_b200.policy import ActorCriticB200
    from opendog_b200.train import GraphedPPOUpdate, ppo_update
    B, S, A = 8192, 33, 8
    g = torch.Generator(device="cuda").manual_seed(1)
    obs = torch.randn(B, S, device="cuda", generator=g); act = torch.randn(B, A, device="cuda", generator=g).clamp(-1, 1)
    logp = torch.randn(B, device="cuda", generator=g) * 0.1 - 8
    adv = torch.randn(B, device="cuda", generator=g); ret = torch.randn(B, device="cuda", generator=g)
    pols, outs = [], []
    for graphed in (False, True):
        pol = ActorCriticB200(S, A, 0.4, seed=0)
        torch.manual_seed(0)
        for p in pol.parameters():
            torch.nn.init.normal_(p, std=0.05)
        opt = torch.optim.Adam(pol.parameters(), lr=1e-3, fused=True, capturable=True)
        if graphed:
            upd = GraphedPPOUpdate(pol, opt, B, S, A, minibatches=4)
            for _ in range(3):                       # first call = capture (its warm-up pass is a real update), then replays
                out = upd(obs, act, logp, adv, ret)
        else:
            for _ in range(3):
                out = ppo_update(pol, opt, obs, act, logp, adv, ret, epochs=1, minibatches=4)
        pols.append(pol); outs.append({k: float(v) for k, v in out.items()})
    for k in outs[0]:
        assert abs(outs[0][k] - outs[1][k]) <= 2e-3 * max(1.0, abs(outs[0][k])), (k, outs)
    for (n0, p0), (_, p1) in zip(pols[0].named_parameters(), pols[1].named_parameters()):
        assert torch.allclose(p0, p1, rtol=0, atol=3e-3), (n0, (p0 - p1).abs().max().item())
    # the tensor-core copy of the weights was refreshed: the rollout-time forward sees the updated parameters
    m0 = pols[0].act(obs[:256], sample=False)[3]; m1 = pols[1].act(obs[:256], sample=False)[3]
    assert torch.allclose(m0, m1, atol=2e-2)


def _tanh_bwd_shapes():
    """(rows, cols) for odg_tanh_backward_bias: every legal width, with rows 1, rp - 1 and 592 * rp * k +- 1 (the edges of the
    per-block row chunks; rp = 2048 / cols rows are in flight per block), where the 4-row unrolled loop starts at 512 and
    256 columns, and the PPO minibatch of configs[3] (65536 x 24 / 4 rows) at both hidden widths."""
    shapes = [(1000, 512), (4097, 256), (37, 1024), (600, 8), (5000, 2048)]
    for cols in (8, 16, 32, 64, 128, 256, 512, 1024, 2048):
        rp = 2048 // cols
        shapes += [(r, cols) for r in sorted({1, rp - 1, 592 * rp - 1, 592 * rp + 1, 592 * rp * 4 - 1, 592 * rp * 4 + 1} - {0})]
    return shapes + [(7105, 512), (14209, 256), (393216, 512), (393216, 256)]


@gpu
@pytest.mark.parametrize("rows,cols", _tanh_bwd_shapes())
def test_tanh_backward_with_bias_gradient_matches_torch(rows, cols):
    """`odg_tanh_backward_bias` (include/odg_policy.h). g = gy * (1 - y*y) is bit-exact against the correctly rounded bf16 of
    the float64 value: y and gy carry 8 significant bits, so y*y, 1 - y*y (|y| >~ 2^-5) and the product are exact in fp32
    with or without FMA contraction, and the only rounding is the final one to bf16. The exception is an element whose
    exact value lies within 2^-22 (relative) of a bf16 rounding midpoint (not on it), where fp32's rounding of a small
    y*y can decide the direction; those are counted and held to one bf16 ulp. torch's own bf16 kernel, which rounds three
    times, stays within a few ulp. The bias gradient is compared with float64 column sums of the kernel's OWN g at the
    fp32 bound of its summation depth (rows per thread + rp + 592 / 8 block partials per slice + 8 slices). Deterministic
    to the bit; nothing written past either output."""
    from opendog_b200 import lib as _lib
    L = _lib.load()
    g_ = torch.Generator(device="cuda").manual_seed(rows + cols)
    gy = torch.randn(rows, cols, device="cuda", generator=g_).to(torch.bfloat16)
    y = torch.tanh(torch.randn(rows, cols, device="cuda", generator=g_) * 2).to(torch.bfloat16)
    scratch = torch.empty(L.odg_tanh_backward_bias_scratch_floats(cols), device="cuda")
    outs = []
    for _ in range(2):
        g, gb = _Guarded((rows, cols), torch.bfloat16, tail=4 * cols), _Guarded((cols,), tail=64)
        _lib.check(L.odg_tanh_backward_bias(_cptr(gy), _cptr(y), _cptr(g.t), _cptr(gb.t), _cptr(scratch), rows, cols,
                                            _stream()), "odg_tanh_backward_bias")
        outs.append((g, gb))
    torch.cuda.synchronize()
    for g, gb in outs:
        g.assert_tail_intact("grad_x"); gb.assert_tail_intact("bias_grad")
    (g, gb), (g2, gb2) = [(a.t, b.t) for a, b in outs]
    assert torch.equal(g.view(torch.int16), g2.view(torch.int16)) and torch.equal(gb.view(torch.int32), gb2.view(torch.int32))
    near_total = 0
    s64 = torch.zeros(cols, dtype=torch.float64, device="cuda"); a64 = torch.zeros_like(s64)
    step = max(1, (1 << 24) // cols)                   # compare in row chunks: a few hundred MB of float64 at a time
    for r0 in range(0, rows, step):
        gyc, yc, gc = gy[r0:r0 + step].double(), y[r0:r0 + step].double(), g[r0:r0 + step]
        exact = gyc * (1.0 - yc * yc)
        ref, dist = _bf16_rn(exact)
        near = (dist > 0) & (dist < 2.0 ** -22)
        near_total += int(near.sum())
        same = gc.view(torch.int16) == ref.to(torch.bfloat16).view(torch.int16)
        bad = ~same & ~near
        assert not bool(bad.any()), (f"{int(bad.sum())} elements differ from the correctly rounded bf16 value, e.g. "
                                     f"gy={gyc[bad][0].item()} y={yc[bad][0].item()} g={gc[bad][0].item()} ref={ref[bad][0].item()}")
        gd = gc.double()
        assert bool(((gd - ref).abs() <= 2 ** -7 * ref.abs())[near].all())           # near a midpoint: one ulp at most
        # torch's own bf16 kernel rounds y*y, 1 - y*y and the product separately: it sits within a few ulp of the above
        tref = torch.ops.aten.tanh_backward(gy[r0:r0 + step], y[r0:r0 + step]).double()
        assert bool(((gd - tref).abs() <= 2 ** -5 * tref.abs() + 2 ** -9 * gyc.abs() + 1e-30).all())
        s64 += gd.sum(0); a64 += gd.abs().sum(0)
    print(f"tanh_backward rows={rows} cols={cols}: {near_total} of {rows * cols} elements within 2^-22 of a bf16 midpoint")
    rp = 2048 // cols
    per_block = -(-rows // 592)
    chunk = -(-per_block // rp) * rp                   # the kernel's rows per block: rounded up to a multiple of rp
    depth = chunk // rp + rp + -(-592 // 8) + 8
    err = (gb.double() - s64).abs()
    assert bool((err <= depth * 2.0 ** -24 * a64).all()), float((err / (a64 * 2.0 ** -24)).max())
    assert L.odg_tanh_backward_bias(_cptr(gy), _cptr(y), _cptr(g), _cptr(gb), _cptr(scratch), rows, 24, None) == -1   # ODG_ERR_INVALID: 24 / 8 = 3
    assert b"odg_tanh_backward_bias" in L.odg_last_error()


@gpu
def test_fused_hidden_layer_backward_matches_autocast_torch():
    """`policy.linear_tanh` (custom backward: one pass for tanh' and the bias gradient) against the plain autocast
    expression it replaces in the PPO update's forward: outputs within one bf16 ulp (hardware tanh), gradients within bf16
    rounding of each other."""
    from opendog_b200.policy import linear_tanh
    torch.manual_seed(5)
    B, K, N = 3000, 48, 512
    x0 = torch.randn(B, K, device="cuda"); w0 = torch.randn(N, K, device="cuda") * 0.1; b0 = torch.randn(N, device="cuda") * 0.1
    go = torch.randn(B, N, device="cuda")
    res = []
    for fused in (False, True):
        x, w, b = (t.clone().requires_grad_(True) for t in (x0, w0, b0))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = linear_tanh(x, w, b) if fused else torch.tanh(torch.nn.functional.linear(x, w, b))
        (y.float() * go).sum().backward()
        res.append((y.detach(), x.grad, w.grad, b.grad))
    (y0, gx0, gw0, gb0), (y1, gx1, gw1, gb1) = res
    # forward: the hardware tanh of the rollout kernel (tanh.approx, rel. error 2^-11) rounded to bf16: within one bf16 ulp
    # of torch's tanhf-based result, the same bits for most elements
    assert y1.dtype == torch.bfloat16
    assert bool(((y1.float() - y0.float()).abs() <= 2 ** -7 * y0.float().abs() + 1e-6).all())
    assert float((y0 == y1).float().mean()) > 0.85
    assert gx1.dtype == torch.float32 and gw1.dtype == torch.float32 and gb1.dtype == torch.float32
    rel = lambda a, b_: float((a - b_).norm() / b_.norm())
    assert rel(gx1, gx0) < 1e-2 and rel(gw1, gw0) < 1e-2 and rel(gb1, gb0) < 1e-2
    # without autocast the plain fp32 / TF32 expression is what runs
    x = x0.clone().requires_grad_(True)
    assert linear_tanh(x, w0, b0).dtype == torch.float32


def _tanh_bf16(x, y, count):
    from opendog_b200 import lib as _lib
    _lib.check(_lib.load().odg_tanh_bf16(_cptr(x), _cptr(y), count, _stream()), "odg_tanh_bf16")


@pytest.fixture(scope="module")
def tanh_table():
    """(every bf16 bit pattern as int16, odg_tanh_bf16 of each as int16 bits), one out-of-place call on all 65536."""
    pats = torch.arange(-32768, 32768, dtype=torch.int32, device="cuda").to(torch.int16)
    x = pats.clone()
    y = _Guarded((65536,), torch.bfloat16)
    _tanh_bf16(x, y.t, 65536)
    torch.cuda.synchronize()
    y.assert_tail_intact("y")
    assert torch.equal(x, pats), "the input of an out-of-place call changed"
    return pats, y.t.view(torch.int16).clone()


@gpu
def test_tanh_bf16_on_every_bf16_value(tanh_table):
    """`odg_tanh_bf16` on all 65536 bf16 values against t64 = torch.tanh in float64 and its correctly rounded bf16 value:
    finite normal x: |y - t64| <= 2^-7 |t64| (bf16 rounding <= 2^-8, tanh.approx.f32 ~2^-11); y = +-1 exactly wherever
    bf16(t64) = +-1, except where |t64| lies within tanh.approx's error (2^-10 relative, taken generously) of the rounding
    midpoint 1 - 2^-9 (|x| in about [3.47, 3.81)), where the relative bound above still holds; +-0 -> 0, +-inf -> +-1,
    NaN -> NaN. bf16 subnormal inputs may come out unchanged or as zero, all of them the same way: on a B200 they come out
    unchanged (tanh.approx.f32 returns these fp32 subnormals as they are), and the 44 inputs of the saturation band
    all give +-1. The in-place call gives the same bits as the out-of-place one."""
    pats, table = tanh_table
    xg = _Guarded((65536,), torch.bfloat16)
    xg.t.view(torch.int16).copy_(pats)
    _tanh_bf16(xg.t, xg.t, 65536)
    torch.cuda.synchronize()
    xg.assert_tail_intact("x (in place)")
    assert torch.equal(xg.t.view(torch.int16), table)
    x = pats.view(torch.bfloat16).double()
    y = table.view(torch.bfloat16).double()
    t64 = torch.tanh(x)
    tb, _ = _bf16_rn(t64)
    expo = (pats.int() >> 7) & 0xFF
    frac = pats.int() & 0x7F
    normal = (expo > 0) & (expo < 255)
    assert bool(((y - t64).abs() <= 2 ** -7 * t64.abs())[normal].all())
    sat = normal & (tb.abs() == 1.0)
    band = sat & (t64.abs() < 1 - 2 ** -10)
    assert bool((y[sat & ~band] == torch.sign(x[sat & ~band])).all())
    print(f"tanh_bf16: {int(band.sum())} inputs within tanh.approx's error of the saturation midpoint, "
          f"{int((y[band].abs() == 1).sum())} of them give +-1")
    zero = (expo == 0) & (frac == 0)
    assert bool((y[zero] == 0).all())
    inf = (expo == 255) & (frac == 0)
    assert bool((y[inf] == torch.sign(x[inf])).all()) and int(inf.sum()) == 2
    nan = (expo == 255) & (frac != 0)
    assert bool(torch.isnan(y[nan]).all()) and not bool(torch.isnan(y[~nan]).any())
    sub = (expo == 0) & (frac != 0)
    kept = bool(torch.equal(table[sub], pats[sub]))
    flushed = bool((y[sub] == 0).all())
    print(f"tanh_bf16: bf16 subnormal inputs {'come out unchanged' if kept else 'flush to zero' if flushed else 'MIXED'}")
    assert kept or flushed


@gpu
@pytest.mark.parametrize("in_place", [False, True])
@pytest.mark.parametrize("count", [8, 24, 65536 + 8, 393216 * 256 + 8, 393216 * 512])
def test_tanh_bf16_matches_the_table_at_every_size(count, in_place, tanh_table):
    """`odg_tanh_bf16` on `count` values tiled from the 65536 bf16 patterns (each tile rotated differently), bit for bit
    against the exhaustive table: counts that are a multiple of 8 but not of 16, and the activations of configs[3]'s PPO
    minibatch (393216 x 512 and x 256, where every thread runs the 4-way unrolled grid-stride loop). Out of place the
    input stays as it was; nothing is written past the output."""
    pats, table = tanh_table
    n_tiles = -(-count // 65536)
    shift = torch.arange(n_tiles, device="cuda", dtype=torch.int64) * 40503 % 65536
    idx = ((torch.arange(65536, device="cuda")[None, :] + shift[:, None]) % 65536).reshape(-1)[:count]
    x_bits = pats[idx]
    expected = table[idx]
    del idx
    y = _Guarded((count,), torch.bfloat16, tail=4096)
    if in_place:
        y.t.view(torch.int16).copy_(x_bits)
        _tanh_bf16(y.t, y.t, count)
    else:
        x = x_bits.clone()
        _tanh_bf16(x, y.t, count)
    torch.cuda.synchronize()
    y.assert_tail_intact("y")
    if not in_place:
        assert torch.equal(x, x_bits), "the input of an out-of-place call changed"
    same = y.t.view(torch.int16) == expected
    assert bool(same.all()), f"{int((~same).sum())} of {count} outputs differ from the table, first at {int((~same).nonzero()[0])}"


# B = 303104 is the last batch whose samples fit one per thread of the 1184-block grid; from 303105 on the grid-stride loop
# runs, and 393216 is the PPO minibatch of configs[3] (65536 x 24 / 4)
_PPO_CASES = [(5000, 8), (333, 12), (70000, 4), (1, 16)] + [(B, A) for B in (303104, 303105, 393216) for A in (1, 3, 8, 16)]


@gpu
@pytest.mark.parametrize("B,A", _PPO_CASES)
def test_fused_ppo_loss_matches_the_torch_expression(B, A):
    """`policy.ppo_loss` on CUDA (odg_ppo_loss: loss terms and gradients in one pass) against the torch expression it
    replaces (the objective of train/train.py:117-130 on the ActorCritic of sim2real/train.py:132-149), autograd in float64:
    loss terms to 1e-5 relative, gradients to 1e-4 of their largest entry; ratios inside and outside the clip range, zero
    advantages, and exact ties (ratio = 1). No sample's ratio lies within 1e-4 of a clip boundary (a float32 ratio on the
    other side of one than the float64 ratio would flip its gradient), so every gradient is checked in full. Two direct
    calls of odg_ppo_loss give the same bits as the autograd path and write nothing past their outputs."""
    from opendog_b200 import lib as _lib
    from opendog_b200.policy import ppo_loss
    g = torch.Generator(device="cuda").manual_seed(B + A)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    mean0, value0, ls0 = torch.tanh(r(B, A)), r(B, 1), (r(1, A) * 0.3 - 0.9)
    action = mean0 + torch.exp(ls0) * r(B, A)
    clip, vf_coef, ent_coef = 0.2, 0.5, 0.005
    with torch.no_grad():
        lp = torch.distributions.Normal(mean0, torch.exp(ls0).expand_as(mean0)).log_prob(action).sum(-1)
        lp64 = torch.distributions.Normal(mean0.double(), torch.exp(ls0.double()).expand_as(mean0)).log_prob(action.double()).sum(-1)
    logp_old = lp + r(B) * 0.25                     # ratios spread over ~[0.5, 2]
    logp_old[::7] = lp[::7]                         # exact ties: ratio = 1
    for _ in range(50):                             # resample the few ratios near a clip boundary
        rt = torch.exp(lp64 - logp_old.double())
        near = ((rt - (1 - clip)).abs() < 1e-4) | ((rt - (1 + clip)).abs() < 1e-4)
        if not bool(near.any()):
            break
        logp_old[near] = lp[near] + r(int(near.sum())) * 0.25
    assert not bool(near.any())
    adv, ret = r(B), r(B)
    adv[::11] = 0.0
    # fused
    m1, v1, l1 = (t.clone().requires_grad_(True) for t in (mean0, value0, ls0))
    loss1, pg1, vf1, ent1 = ppo_loss(m1, v1, l1, action, logp_old, adv, ret, clip, vf_coef, ent_coef)
    loss1.backward()
    # torch, float64
    m2, v2, l2 = (t.double().clone().requires_grad_(True) for t in (mean0, value0, ls0))
    d = torch.distributions.Normal(m2, torch.exp(l2.expand_as(m2)), validate_args=False)
    logp = d.log_prob(action.double()).sum(-1)
    ratio = torch.exp(logp - logp_old.double())
    a = adv.double()
    pg2 = -torch.min(ratio * a, torch.clamp(ratio, 1 - clip, 1 + clip) * a).mean()
    vf2 = torch.nn.functional.mse_loss(v2.squeeze(-1), ret.double())
    ent2 = d.entropy().sum(-1).mean()
    loss2 = pg2 + vf_coef * vf2 - ent_coef * ent2
    loss2.backward()
    for x, y in ((loss1, loss2), (pg1, pg2), (vf1, vf2), (ent1, ent2)):
        x, y = float(x.detach()), float(y.detach())
        assert abs(x - y) <= 1e-5 * (1 + abs(y)), (x, y)
    assert float((m1.grad.double() - m2.grad).abs().max()) <= 1e-4 * float(m2.grad.abs().max()) + 1e-12
    assert float((v1.grad.double() - v2.grad).abs().max()) <= 1e-5 * float(v2.grad.abs().max()) + 1e-12
    assert float((l1.grad.double() - l2.grad).abs().max()) <= 1e-4 * float(l2.grad.abs().max()) + 1e-9
    assert m1.grad.shape == mean0.shape and v1.grad.shape == value0.shape and l1.grad.shape == ls0.shape
    # the C ABI directly, twice, into guard-banded outputs
    L = _lib.load()
    scratch = torch.empty(L.odg_ppo_loss_scratch_floats(), device="cuda")
    ins = [t.contiguous() for t in (mean0, value0.reshape(-1), ls0.reshape(-1), action, logp_old, adv, ret)]
    runs = []
    for _ in range(2):
        o = {"loss": _Guarded((1,)), "terms": _Guarded((4,)), "g_mean": _Guarded((B, A)), "g_value": _Guarded((B,)),
             "g_log_std": _Guarded((A,))}
        _lib.check(L.odg_ppo_loss(*(_cptr(t) for t in ins), B, A, clip, vf_coef, ent_coef,
                                  *(_cptr(o[k].t) for k in ("loss", "terms", "g_mean", "g_value", "g_log_std")),
                                  _cptr(scratch), _stream()), "odg_ppo_loss")
        runs.append(o)
    torch.cuda.synchronize()
    bits = lambda t: t.detach().reshape(-1).view(torch.int32)
    autograd = {"loss": loss1, "terms": torch.stack([loss1, pg1, vf1, ent1]), "g_mean": m1.grad, "g_value": v1.grad,
                "g_log_std": l1.grad}
    for k, ref in autograd.items():
        for o in runs:
            o[k].assert_tail_intact(k)
            assert torch.equal(bits(o[k].t), bits(ref)), k


@gpu
def test_fused_ppo_loss_with_infinite_clip_is_the_sim2real_update():
    """sim2real/train.py:566-569: actor_loss = -(log_prob * adv).mean(), critic MSE, entropy — the clipped objective with
    clip = +inf and logp_old = logp (ratio 1): same loss gradients from `policy.ppo_loss`."""
    from opendog_b200.policy import ppo_loss
    g = torch.Generator(device="cuda").manual_seed(77)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    B, A = 4000, 8
    mean0, value0, ls0 = torch.tanh(r(B, A)), r(B, 1), (r(1, A) * 0.3 - 0.9)
    action = mean0 + torch.exp(ls0) * r(B, A)
    adv, ret = r(B), r(B)
    VALUE_LOSS_COEF, ENT = 0.5, 0.01
    m2, v2, l2 = (t.double().clone().requires_grad_(True) for t in (mean0, value0, ls0))
    d = torch.distributions.Normal(m2, torch.exp(l2.expand_as(m2)), validate_args=False)
    logp = d.log_prob(action.double()).sum(-1)
    # (the reference takes entropy().mean() over [B, A]; per-dimension mean = the summed entropy / A)
    loss2 = -(logp * adv.double()).mean() + VALUE_LOSS_COEF * torch.nn.functional.mse_loss(v2.squeeze(-1), ret.double()) \
        - ENT * d.entropy().mean()
    loss2.backward()
    m1, v1, l1 = (t.clone().requires_grad_(True) for t in (mean0, value0, ls0))
    loss1, _, _, _ = ppo_loss(m1, v1, l1, action, logp.detach().float(), adv, ret, float("inf"), VALUE_LOSS_COEF, ENT / A)
    loss1.backward()
    for a_, b_ in ((m1.grad, m2.grad), (v1.grad, v2.grad), (l1.grad, l2.grad)):
        assert float((a_.double() - b_).abs().max()) <= 2e-4 * float(b_.abs().max()) + 1e-12
