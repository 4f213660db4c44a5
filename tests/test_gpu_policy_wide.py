"""GPU tests of the terrain trainer's policy forward (`k_mlp_wide`: 1024 / 512 hidden, sim2real/train2.py:149-157) and of
on-device rollouts of both QuadrupedEnv trainers through `opendog_b200.rollout.Rollout`.

The forward is checked against `_kernel_model`, a torch restatement of the kernel's own contract: bf16 inputs and
weights, exact (float64) dot products, fp32 bias, the SAME hardware tanh.approx.f32 on the hidden layers (compiled at
run time with torch's jiterator), every hidden activation rounded to bf16, fp32 head and tanh on the actor output.
What is left between kernel and model is the kernel's fp32 accumulation order. It moves a pre-activation by about 2^-24
of its sum of absolute products, which changes the bf16 rounding of a hidden activation only when that activation lies
that close to a rounding midpoint: a rare one-ulp flip in a few of the 1536 hidden units of a row. MODEL_TOL and
MODEL_RMS_TOL bound that: see their comment for the measurement behind them and what they reject. Against the plain fp32 torch module the kernel stays
within the 3e-2 of the 512 / 256 tests (bf16 quantisation)."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from test_gpu_policy import _Guarded, _ref_forward, _sample_eps_np  # noqa: E402

H = (1024, 512)
# |kernel - _kernel_model| of the actor mean and of the value (relative to max(1, |value|)): the largest over a call and the
# root mean square over its rows and outputs. Measured on an NVIDIA B200 (1000 W power limit) over the cases below: max
# up to 6.1e-4 (a row whose hidden activations had several accumulation-order flips), rms 9e-6 to 2.4e-5. Kernels that
# break the contract, built and run against these tests on the same card: tanhf instead of tanh.approx in the hidden
# epilogues gives rms 1.3e-4 to 1.6e-4 on every multi-row case (max up to 1.2e-3); hidden 2 left in fp32 before the head
# gives rms 4.4e-4 to 4.9e-4 (max 7e-4 to 2.4e-3). MODEL_RMS_TOL sits at twice the largest measured rms and 2.6 times
# below the smallest rms of either broken kernel; MODEL_TOL at 2.5 times the largest measured max.
MODEL_TOL = 1.5e-3
MODEL_RMS_TOL = 5e-5
# |log(pi_update / pi_rollout)| per sample: a quarter of PPO's clip range of 0.2, so numerics alone clip no sample in the
# first epoch. Measured on the same card: max 0.020, rms 0.0025 over 8192 samples x 8 dims.
LOGP_TOL = 5e-2


def _wide_policy(S, A, seed=7, hidden=H, scale=2.0, torch_seed=None):
    from opendog_b200.policy import ActorCriticB200
    torch.manual_seed(S * 100 + A if torch_seed is None else torch_seed)
    m = ActorCriticB200(S, A, 0.4, seed=seed, hidden=hidden)
    with torch.no_grad():
        for p in m.parameters():
            if p.dim() == 2 and p.shape[0] > 16:
                p.mul_(scale)                    # push hidden units into the non-linear range of tanh
        m.action_log_std.copy_(torch.linspace(-1.5, -0.5, A)[None])
    m.sync_weights()
    return m


_TANH_APPROX = []


def _tanh_approx(x):
    """tanh.approx.f32 (the instruction the kernels' hidden-layer epilogues use) elementwise on a float32 CUDA tensor."""
    if not _TANH_APPROX:
        _TANH_APPROX.append(torch.cuda.jiterator._create_jit_fn(
            'template <typename T> T tanh_approx(T x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"((float)x)); return y; }'))
    return _TANH_APPROX[0](x.float().contiguous())


def _kernel_model(m, obs, params=None):
    """(mean [N, A], value [N]) of the kernel's contract, in torch; `params` = the module's parameters in
    `m.parameters()` order (default: the current ones)."""
    P = dict(zip([n for n, _ in m.named_parameters()], params if params is not None else [p.detach() for p in m.parameters()]))
    bf = lambda t: t.to(torch.bfloat16).to(torch.float64)

    def run(net):
        x = bf(obs)
        for i in (0, 2):
            z = (x @ bf(P[f"{net}.{i}.weight"]).T).float() + P[f"{net}.{i}.bias"].float()
            x = bf(_tanh_approx(z))
        return (x @ bf(P[f"{net}.4.weight"]).T).float() + P[f"{net}.4.bias"].float()
    return torch.tanh(run("actor")), run("critic")[:, 0]


def _ref_forward_params(m, obs, params):
    """tests/test_gpu_policy.py's bf16-rounding reference forward on the given parameter list."""
    import copy
    import types
    c = types.SimpleNamespace(actor=copy.deepcopy(m.actor), critic=copy.deepcopy(m.critic))
    P = dict(zip([n for n, _ in m.named_parameters()], params))
    with torch.no_grad():
        for net in ("actor", "critic"):
            for n, p in getattr(c, net).named_parameters():
                p.copy_(P[f"{net}.{n}"])
    return _ref_forward(c, obs, True)


def _model_gap(mean, value, r_mean, r_val):
    """(max, root mean square) over rows and outputs of |kernel - model|: mean absolute, value relative to max(1, |value|)."""
    d = torch.cat([(mean - r_mean).reshape(-1), ((value - r_val) / r_val.abs().clamp_min(1.0)).reshape(-1)]).double()
    return d.abs().max().item(), d.square().mean().sqrt().item()


def _waves():
    return 128 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# n: a row, a partial CTA, one CTA, one CTA + 1, about one wave W (one 128-row CTA per SM) and W + 1, 65537. W and W + 1 are
# approximate wave edges: CTAs run in 2-CTA clusters and cluster placement may leave SMs idle. 65537 rows (3.5 waves)
# is what makes CTAs follow others on the same SM (TMEM alloc / dealloc, mbarrier init).
_CASES = [(12, 8, n) for n in (1, 127, 128, 129, "W", "W+1", 65537)]
_CASES += [(S, A, 257) for S in (1, 12, 16, 17, 64) for A in (1, 8, 16)]


@pytest.mark.parametrize("S,A,N", _CASES)
def test_wide_forward_matches_torch_and_samples_the_keyed_stream(S, A, N):
    if isinstance(N, str):
        N = _waves() + (1 if N == "W+1" else 0)
    m = _wide_policy(S, A)
    first_row = 3 * 65536 + 5
    obs = torch.randn(N, S, device="cuda") * 1.5
    out = {"mean": _Guarded((N, A), tail=128 * A), "action": _Guarded((N, A), tail=128 * A),
           "value": _Guarded((N,)), "logp": _Guarded((N,))}
    action, logp, value, mean = m.act(obs, step=3, first_row_id=first_row, out={k: g.t for k, g in out.items()})
    torch.cuda.synchronize()
    for k, g in out.items():
        g.assert_tail_intact(k)
    # mean / value against the kernel's contract restated in torch; against the fp32 module within 3e-2
    r_mean, r_val = _kernel_model(m, obs)
    gap, rms = _model_gap(mean, value, r_mean, r_val)
    print(f"wide forward S={S} A={A} N={N}: gap to the model max {gap:.3g} rms {rms:.3g}")
    assert gap <= MODEL_TOL and rms <= MODEL_RMS_TOL, (gap, rms)
    f_mean, f_val = _ref_forward(m, obs, False)
    assert (mean - f_mean).abs().max().item() < 3e-2
    assert (value - f_val).abs().max().item() < 3e-2 * max(1.0, f_val.abs().max().item())
    # every row's noise against the numpy Philox / Box-Muller restatement: action to fp32 rounding (expf, logf, sqrtf,
    # sincosf are within 2 ulp; the sincos argument 2 pi u2 is rounded once), logp to the fp32 sum of A terms
    ls = m.action_log_std.detach().cpu().double().numpy().reshape(-1)
    sig = np.exp(ls)
    act = action.cpu().double().numpy(); mu = mean.cpu().double().numpy(); lp = logp.cpu().double().numpy()
    eps = _sample_eps_np(7, first_row + np.arange(N, dtype=np.uint64), 3, A)
    tol_a = 2.0 ** -21 * (np.abs(mu) + sig * (np.abs(eps) + 6.0))
    assert bool((np.abs(act - (mu + sig * eps)) <= tol_a).all())
    terms = -0.5 * eps ** 2 - ls - 0.5 * math.log(2 * math.pi)
    tol_l = 2.0 ** -20 * np.sum(np.abs(terms) + eps ** 2 * 6.0, axis=1) + A * 2.0 ** -22 * np.abs(terms).sum(1)
    assert bool((np.abs(lp - terms.sum(1)) <= tol_l + 1e-6).all())
    # deterministic path and repeatability: the same call twice gives the same bits
    a2, lp2, v2, mean2 = m.act(obs, sample=False)
    assert lp2 is None and torch.equal(a2, mean2) and torch.equal(mean2, mean) and torch.equal(v2, value)
    a3, lp3, v3, m3 = m.act(obs, step=3, first_row_id=first_row)
    assert torch.equal(a3, action) and torch.equal(lp3, logp) and torch.equal(v3, value)


@pytest.mark.parametrize("A", [1, 8, 16])
def test_wide_and_narrow_kernels_draw_the_same_noise(A):
    """With the actor head zeroed, mean = tanh(0) = 0 in both kernels, so action = exp(log_std) * eps and logp are the
    noise alone: the 1024 / 512 and the 512 / 256 kernel must give the same bits for the same (seed, row, step) key."""
    S, N = 12, 3000
    outs = []
    for hidden in (H, (512, 256)):
        m = _wide_policy(S, A, seed=99, hidden=hidden)
        with torch.no_grad():
            m.actor[4].weight.zero_(); m.actor[4].bias.zero_()
        m.sync_weights()
        obs = torch.randn(N, S, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
        a, lp, _, mean = m.act(obs, step=11, first_row_id=4096)
        assert torch.equal(mean, torch.zeros_like(mean))
        outs.append((a.clone(), lp.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_wide_rows_split_over_calls_and_the_device_step_counter():
    S, A, N, k = 12, 8, 5000, 1931
    m = _wide_policy(S, A)
    obs = torch.randn(N, S, device="cuda")
    full = [t.clone() for t in m.act(obs, step=5, first_row_id=100)]
    lo = m.act(obs[:k].clone(), step=5, first_row_id=100)
    lo = [t.clone() for t in lo]
    hi = m.act(obs[k:].clone(), step=5, first_row_id=100 + k)
    for f, a, b in zip(full, lo, hi):
        assert torch.equal(f, torch.cat([a, b]))
    base = torch.tensor([5], dtype=torch.int32, device="cuda")
    via_dev = m.act(obs, step=0, step_base=base, first_row_id=100)
    assert all(torch.equal(f, g) for f, g in zip(full, via_dev))
    base.fill_(6)
    moved = m.act(obs, step=0, step_base=base, first_row_id=100)
    assert not torch.equal(moved[0], full[0]) and torch.equal(moved[3], full[3])


def test_logp_old_matches_the_update_phase_forward():
    """The rollout's logp (kernel) against the log-prob the PPO update computes from `forward_padded` under bf16 autocast
    on the same rows: every |log ratio| within LOGP_TOL. The update phase rounds each pre-activation to bf16 before its
    tanh.approx (the autocast GEMM's output), which the kernel does not; that is most of the gap, and it is larger than
    the difference between tanh.approx and tanhf, so this comparison cannot tell the two apart: the forward test against
    `_kernel_model` holds the kernel to tanh.approx."""
    from opendog_b200.compat import BatchedTerrainQuadrupedEnv
    from opendog_b200.rollout import Rollout
    env = BatchedTerrainQuadrupedEnv(1024, seed=3, auto_reset=True, max_steps=40)
    m = _wide_policy(12, 8, seed=5, scale=1.0)
    ro = Rollout(env, m, horizon=8, use_graph=False)
    ro.collect()
    obs = ro.obs[:ro.T].reshape(-1, 12)
    act = ro.action.reshape(-1, 8)
    lp_k = ro.logp.reshape(-1).double()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        d, _ = m.forward_padded(m.pad_obs(obs.to(torch.bfloat16)))
    lp_u = d.log_prob(act).float().sum(-1).double()
    gap = (lp_u - lp_k).abs()
    print(f"logp_old: max |log ratio| {gap.max().item():.3g}, 99.9th percentile {gap.quantile(0.999).item():.3g}, "
          f"rms {gap.square().mean().sqrt().item():.3g}")
    assert gap.max().item() <= LOGP_TOL


# ---- rollouts of the two QuadrupedEnv trainers --------------------------------------------------------------------------
_VARIANTS = {"train": ((22, 4), (512, 256)), "terrain": ((12, 8), H)}


def _make(variant, N, first_env_id=0, seed=0):
    from opendog_b200.compat import BatchedQuadrupedEnv, BatchedTerrainQuadrupedEnv
    from opendog_b200.policy import ActorCriticB200
    (S, A), hidden = _VARIANTS[variant]
    if variant == "terrain":
        env = BatchedTerrainQuadrupedEnv(N, seed=4, first_env_id=first_env_id, auto_reset=True, max_steps=5)
    else:
        env = BatchedQuadrupedEnv(N, first_env_id=first_env_id, auto_reset=True, max_steps=5)
    torch.manual_seed(seed)
    pol = ActorCriticB200(S, A, 0.4, seed=13, hidden=hidden)
    return env, pol


def _buffers(ro, env):
    out = [ro.obs, ro.action, ro.logp, ro.value, ro.reward, ro.terminated, ro.truncated, ro.done]
    if hasattr(env, "hfield_data"):
        out.append(env.hfield_data)
    return [x.clone() for x in out]


def _collect3(variant, N, use_graph, first_env_id=0):
    from opendog_b200.rollout import Rollout
    env, pol = _make(variant, N, first_env_id)
    ro = Rollout(env, pol, horizon=8, use_graph=use_graph, first_row_id=first_env_id)
    fields = []
    for _ in range(3):
        if hasattr(env, "hfield_data"):
            fields.append(env.hfield_data.clone())
        ro.collect()
    torch.cuda.synchronize()
    return env, pol, ro, fields


@pytest.mark.parametrize("variant", ["train", "terrain"])
def test_quadruped_rollout_graphed_eager_hand_loop_and_shards(variant):
    """Graphed == eager, bit for bit, over three horizons (warm-up, capture + first replay, replay); both equal a
    hand-written `act` + `step` loop; N environments equal two shards of N / 2 with first_env_id / first_row_id offsets,
    terrain fields included; terminated / truncated agree with the termination reason; the fields of the environments that
    finished during the replayed horizon were regenerated inside the graph."""
    N, T = 256, 8
    env_e, _, ro_e, _ = _collect3(variant, N, False)
    eager = _buffers(ro_e, env_e)
    env_g, _, ro_g, fields = _collect3(variant, N, True)
    assert ro_g.graph is not None
    graphed = _buffers(ro_g, env_g)
    for a, b in zip(eager, graphed):
        assert torch.equal(a, b)
    done_last = ro_g.done.any(0)
    assert bool(done_last.all()), "max_steps = 5 ends every episode inside a horizon of 8"
    if variant == "terrain":
        changed = (graphed[-1] != fields[2]).any(1)
        assert changed.float().mean().item() > 0.3, "fields regenerated inside the replayed graph"
    # hand-written loop: the same kernels called one by one, with env.step and the reason it reports
    env, pol = _make(variant, N)
    obs = env.reset().clone()
    for h in range(3):
        step0 = h * (T + 1)
        rows = dict(obs=[obs], action=[], logp=[], value=[], reward=[], term=[], trunc=[])
        for t in range(T):
            a, lp, v, _ = pol.act(obs, sample=True, step=step0 + t)
            o, r, d, info = env.step(a)
            reason = info["termination_reason"]
            term = (reason != 0).to(torch.uint8); trunc = (d & (reason == 0)).to(torch.uint8)
            assert torch.equal(d, (term | trunc).bool())
            obs = o.clone()
            for k, x in (("obs", obs), ("action", a), ("logp", lp), ("value", v), ("reward", r), ("term", term), ("trunc", trunc)):
                rows[k].append(x.clone())
        _, _, vT, _ = pol.act(obs, sample=False, step=step0 + T)
        rows["value"].append(vT.clone())
    hand = [torch.stack(rows[k]) for k in ("obs", "action", "logp", "value", "reward", "term", "trunc")]
    for a, b in zip(hand, eager[:7]):
        assert torch.equal(a, b)
    if variant == "terrain":
        assert torch.equal(env.hfield_data, eager[-1])
    # terminated / truncated against the reason of the last step, and done = terminated | truncated
    assert torch.equal(eager[7], eager[5] | eager[6]) and not bool((eager[5] & eager[6]).any())
    # two shards of N / 2
    parts = [_buffers(ro, e) for e, _, ro, _ in (_collect3(variant, N // 2, True, f) for f in (0, N // 2))]
    for i, full in enumerate(eager):
        dim = 0 if i == len(eager) - 1 and variant == "terrain" else 1
        assert torch.equal(full, torch.cat([parts[0][i], parts[1][i]], dim=dim)), i


@pytest.mark.parametrize("variant", ["train", "terrain"])
def test_quadruped_training_iteration(variant):
    """collect -> advantages -> GraphedPPOUpdate (which re-packs the weights) -> the kernel's forward on the updated weights
    matches the bf16 torch model within the derived bound."""
    from opendog_b200.rollout import Rollout
    from opendog_b200.train import GraphedPPOUpdate
    N, T = 512, 8
    env, pol = _make(variant, N)
    S, A = env.obs_dim, env.act_dim
    ro = Rollout(env, pol, horizon=T, use_graph=True)
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3, fused=True, capturable=True)
    upd = GraphedPPOUpdate(pol, opt, N * T, S, A, minibatches=4)
    before = [p.detach().clone() for p in pol.parameters()]
    for _ in range(2):
        ro.collect()
        adv, ret, _ = ro.advantages(normalize=True, group=False)
        out = upd(ro.obs[:T].reshape(-1, S), ro.action.reshape(-1, A), ro.logp.reshape(-1), adv.reshape(-1), ret.reshape(-1))
        assert all(math.isfinite(float(v)) for v in out.values())
    assert any(not torch.equal(a, b) for a, b in zip(before, pol.parameters()))
    obs = ro.obs[T].clone()
    mean, _, value, _ = pol.act(obs, sample=False)
    if pol.hidden == H:
        gap, rms = _model_gap(mean, value, *_kernel_model(pol, obs))
        stale, _ = _model_gap(mean, value, *_kernel_model(pol, obs, before))
        print(f"after the update: gap to the model max {gap:.3g} rms {rms:.3g}, to the model on the weights before it {stale:.3g}")
        assert gap <= MODEL_TOL and rms <= MODEL_RMS_TOL
        assert stale > 10 * MODEL_TOL                           # the forward runs on the updated weights, not stale ones
    else:
        r_mean, r_val = _ref_forward(pol, obs, True)         # the 512 / 256 kernel's tolerances (tests/test_gpu_policy.py)
        assert (mean - r_mean).abs().max().item() < 4e-3
        assert (value - r_val).abs().max().item() < 4e-3 * max(1.0, r_val.abs().max().item())
        s_mean, s_val = _ref_forward_params(pol, obs, before)
        assert max((mean - s_mean).abs().max().item(), (value - s_val).abs().max().item()) > 4e-2
