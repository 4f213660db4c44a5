"""GPU tests of batched MPPI (include/odg_mppi.h "Batched MPPI", opendog_b200.mppi.BatchedMPPI). The oracle is the
single-robot path: group g of a K-robot plan must equal, bit for bit, a single-robot plan with seed + g on an S-sample
handle that odg_mppi_broadcast filled from robot g; the closed loop must equal the same steps done by hand."""
import ctypes as C
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

INVALID = -1
SEED = 0xFFFFFFFE            # seed + g crosses 2**32 from g = 2: the 64-bit key carries into its high word


def p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _lib():
    from opendog_b200 import lib
    return lib, lib.load()


def _tilt(q, i, deg):
    """Robot i's trunk rolled by `deg` degrees (MuJoCo quaternion w, x, y, z at qpos[3:7])."""
    h = math.radians(deg) / 2
    q[i, 3:7] = torch.tensor([math.cos(h), math.sin(h), 0.0, 0.0], device=q.device)


def _robots(K, model="our_robot", steps=12, tilt=None, seed=3, **cfg):
    """K robots that have landed and walk under small random actions (so their warm starts are nonzero); robot `tilt`
    is then rolled 35 degrees, past the +-15 degree termination band, and all take one more step (with auto_reset = 0
    the tilted robot stays tilted)."""
    from opendog_b200.env import BatchedWalkEnv
    r = BatchedWalkEnv(K, model=model, seed=seed, info_keys=None, **cfg)
    r.reset()
    g = torch.Generator(device="cuda").manual_seed(seed)
    act = lambda: torch.rand(K, r.act_dim, device="cuda", generator=g) * 0.6 - 0.3
    for _ in range(steps):
        r.step(act())
    if tilt is not None:
        q, v = r.get_state()
        _tilt(q, tilt, 35.0)
        r.set_state(q, v)
        r.step(act())
        assert bool(r.terminated[tilt])
    torch.cuda.synchronize()
    return r


def _samples(n, model="our_robot", **cfg):
    from opendog_b200.env import BatchedWalkEnv
    return BatchedWalkEnv(n, model=model, seed=11, info_keys=None, auto_reset=0, **cfg)


def _broadcast(samples, robots, first, groups):
    lib, L = _lib()
    lib.check(L.odg_mppi_broadcast(samples._h, robots._h, first, groups, None), "odg_mppi_broadcast")


# ---------------------------------------------------------------------------------------------------- broadcast
def test_broadcast_copies_every_robot_into_its_group():
    K, S = 4, 5
    robots = _robots(K, auto_reset=0)
    q, v = robots.get_state()
    es = robots.get_env_state()
    assert (es["step"] > 0).all() and es["last_action"].abs().sum() > 0
    for first, groups in ((0, K), (1, 2), (3, 1)):
        smp = _samples(groups * S)
        _broadcast(smp, robots, first, groups)
        sq, sv = smp.get_state()
        ses = smp.get_env_state()
        torch.cuda.synchronize()
        sel = slice(first, first + groups)
        assert torch.equal(sq, q[sel].repeat_interleave(S, 0)) and torch.equal(sv, v[sel].repeat_interleave(S, 0))
        for k in es:
            assert torch.equal(ses[k], es[k][sel].repeat_interleave(S, 0)), (first, groups, k)


@pytest.mark.parametrize("model", ["our_robot", "go1"])
def test_broadcast_sample_steps_like_its_robot_bit_for_bit(model):
    """Robots mid-stride with nonzero warm starts: a sample stepped with its robot's action reproduces the robot's own
    step exactly, so the warm start and the env-side state travel with qpos / qvel."""
    from opendog_b200.env import BatchedWalkEnv
    K, S = 3, 7
    robots = BatchedWalkEnv(K, model=model, seed=5, info_keys=("qacc",), auto_reset=0)
    robots.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    A = robots.act_dim
    for _ in range(14):
        robots.step(torch.rand(K, A, device="cuda", generator=g) * 0.6 - 0.3)
    assert robots.info["qacc"].abs().amax(1).min().item() > 0          # the warm start of the next solve is nonzero
    smp = _samples(K * S, model=model)
    _broadcast(smp, robots, 0, K)
    act = torch.rand(K, A, device="cuda", generator=g) * 0.6 - 0.3
    for _ in range(3):
        robots.step(act)
        smp.step(act.repeat_interleave(S, 0).contiguous())
        rq, rv = robots.get_state()
        sq, sv = smp.get_state()
        torch.cuda.synchronize()
        rep = lambda t: t.repeat_interleave(S, 0)
        assert torch.equal(sq, rep(rq)) and torch.equal(sv, rep(rv))
        assert torch.equal(smp.obs, rep(robots.obs)) and torch.equal(smp.reward, rep(robots.reward))


def test_broadcast_refusals_issue_no_device_work():
    lib, L = _lib()
    from opendog_b200.env import BatchedWalkEnv
    robots = BatchedWalkEnv(4, info_keys=None)
    smp = _samples(12)
    go1 = _samples(12, model="go1")
    go1_robots = BatchedWalkEnv(2, model="go1", info_keys=None)
    jump = _samples(12, model="go1", task="jump")
    auto = BatchedWalkEnv(12, info_keys=None)                         # auto_reset = 1
    ten = _samples(10)
    handles = (robots, smp, go1, go1_robots, jump, auto, ten)
    before = [h.launch_count for h in handles]
    cases = [((None, robots._h, 0, 1), b"null handle"), ((smp._h, None, 0, 1), b"null handle"),
             ((go1._h, robots._h, 0, 2), b"nq / nv / nu / task"), ((jump._h, go1_robots._h, 0, 2), b"nq / nv / nu / task"),
             ((smp._h, robots._h, 0, 0), b"out of range"), ((smp._h, robots._h, 0, -1), b"out of range"),
             ((smp._h, robots._h, 3, 2), b"out of range"), ((smp._h, robots._h, -1, 2), b"out of range"),
             ((smp._h, robots._h, 0, 5), b"out of range"),
             ((ten._h, robots._h, 0, 4), b"whole number of groups"),
             ((auto._h, robots._h, 0, 4), b"auto_reset = 0")]
    for args, msg in cases:
        assert L.odg_mppi_broadcast(*args, None) == INVALID and msg in L.odg_last_error(), (args, msg)
    m = torch.zeros(4, 2, 8, device="cuda"); a = torch.zeros(2, 12, 8, device="cuda"); c = torch.zeros(12, device="cuda")
    assert L.odg_mppi_rollout_groups(smp._h, 5, p(m), 0.3, 2, 0, 0, None, 100.0, p(a), p(c), None) == INVALID
    assert b"whole number of groups" in L.odg_last_error()
    assert L.odg_mppi_rollout_groups(smp._h, 0, p(m), 0.3, 2, 0, 0, None, 100.0, p(a), p(c), None) == INVALID
    assert L.odg_mppi_rollout_groups(auto._h, 4, p(m), 0.3, 2, 0, 0, None, 100.0, p(a), p(c), None) == INVALID
    assert b"auto_reset = 0" in L.odg_last_error()
    assert [h.launch_count for h in handles] == before
    if torch.cuda.device_count() > 1:
        other = BatchedWalkEnv(4, device="cuda:1", info_keys=None)
        assert L.odg_mppi_broadcast(smp._h, other._h, 0, 4, None) == INVALID and b"different devices" in L.odg_last_error()


# ---------------------------------------------------------------------------------------------------- group equivalence
def _single_plans(robots, K, S, T, mean, iteration, model="our_robot", lam=0.8):
    """K single-robot plans: an S-sample handle filled from robot g, odg_mppi_rollout(seed + g), odg_mppi_reduce."""
    lib, L = _lib()
    one = _samples(S, model=model)
    A = one.act_dim
    acts, costs, means, stats = [], [], [], []
    for g in range(K):
        _broadcast(one, robots, g, 1)
        a = torch.empty(T, S, A, device="cuda"); c = torch.empty(S, device="cuda")
        nm = torch.empty(T, A, device="cuda"); st = torch.empty(4, device="cuda")
        lib.check(L.odg_mppi_rollout(one._h, p(mean[g]), 0.3, T, C.c_uint64(SEED + g), iteration, None, 100.0, p(a), p(c), None),
                  "odg_mppi_rollout")
        lib.check(L.odg_mppi_reduce(p(c), p(a), T, S, A, lam, p(nm), p(st), None), "odg_mppi_reduce")
        acts.append(a); costs.append(c); means.append(nm); stats.append(st)
    torch.cuda.synchronize()
    return torch.cat(acts, 1), torch.cat(costs), torch.stack(means), torch.stack(stats)


def _check_groups(K, S, T, model="our_robot", lam=0.8, **shape):
    lib, L = _lib()
    robots = _robots(K, model=model, tilt=K // 2 if K > 1 else None, auto_reset=0)
    A = robots.act_dim
    g = torch.Generator(device="cuda").manual_seed(K * 1000 + S * 10 + T)
    mean = (torch.rand(K, T, A, device="cuda", generator=g) - 0.5).contiguous()
    smp = _samples(K * S, model=model, **shape)
    N = K * S
    acts = torch.full((T, N, A), float("nan"), device="cuda"); cost = torch.full((N,), float("nan"), device="cuda")
    nm = torch.empty(K, T, A, device="cuda"); st = torch.empty(K, 4, device="cuda")
    _broadcast(smp, robots, 0, K)
    lib.check(L.odg_mppi_rollout_groups(smp._h, K, p(mean), 0.3, T, C.c_uint64(SEED), 3, None, 100.0, p(acts), p(cost), None),
              "odg_mppi_rollout_groups")
    lib.check(L.odg_mppi_reduce_groups(p(cost), p(acts), T, K, S, A, lam, p(nm), p(st), None), "odg_mppi_reduce_groups")
    ra, rc, rm, rs = _single_plans(robots, K, S, T, mean, 3, model=model, lam=lam)
    assert torch.equal(acts, ra) and torch.equal(cost, rc), (K, S, T, shape)
    assert torch.equal(nm, rm) and torch.equal(st, rs), (K, S, T, shape)
    if K > 1:            # the tilted robot's samples all terminate inside the horizon and pay the termination cost
        assert (cost[(K // 2) * S:(K // 2 + 1) * S] > 50).all()
    return cost


@pytest.mark.parametrize("shape", [dict(launch_lanes=8, launch_fat=0), dict(launch_lanes=32, launch_fat=1)],
                         ids=["lanes8_lean", "lanes32_fat"])
def test_groups_equal_single_robot_plans(shape):
    for K in (1, 3, 7):
        for S in (1, 37, 128):
            for T in (1, 10):
                _check_groups(K, S, T, **shape)


def test_groups_equal_single_robot_plans_beyond_one_wave():
    _check_groups(16, 1024, 4)


def test_groups_equal_single_robot_plans_go1():
    _check_groups(3, 37, 10, model="go1")


# ---------------------------------------------------------------------------------------------------- reduction
def test_reduce_groups_equal_reduce_on_each_slice():
    lib, L = _lib()
    gen = torch.Generator().manual_seed(0)
    for G, S, T, A in ((1, 1000, 7, 8), (5, 300, 7, 8), (3, 37, 4, 12), (2, 12000, 3, 8)):
        N = G * S
        cost = (torch.randn(N, generator=gen) * 3 + 5).cuda()
        act = (torch.rand(T, N, A, generator=gen) * 2 - 1).cuda()
        out = torch.empty(G, T, A, device="cuda"); st = torch.empty(G, 4, device="cuda")
        lib.check(L.odg_mppi_reduce_groups(p(cost), p(act), T, G, S, A, 0.7, p(out), p(st), None), "odg_mppi_reduce_groups")
        for g in range(G):
            c = cost[g * S:(g + 1) * S].contiguous(); a = act[:, g * S:(g + 1) * S].contiguous()
            o1 = torch.empty(T, A, device="cuda"); s1 = torch.empty(4, device="cuda")
            lib.check(L.odg_mppi_reduce(p(c), p(a), T, S, A, 0.7, p(o1), p(s1), None), "odg_mppi_reduce")
            torch.cuda.synchronize()
            assert torch.equal(out[g], o1) and torch.equal(st[g], s1), (G, S, g)
            cd = c.double().cpu().numpy(); w = np.exp(-(cd - cd.min()) / 0.7)
            ref = np.einsum("n,tna->ta", w, a.double().cpu().numpy()) / w.sum()
            assert np.abs(out[g].cpu().numpy() - ref).max() < 2e-5
            assert int(st[g, 3].item()) == int(cd.argmin())              # argmin within the group
    cost = torch.zeros(2 * 12001, device="cuda"); act = torch.zeros(1, 2 * 12001, 8, device="cuda")
    out = torch.empty(2, 1, 8, device="cuda")
    assert L.odg_mppi_reduce_groups(p(cost), p(act), 1, 2, 12001, 8, 1.0, p(out), None, None) == INVALID
    assert b"12000" in L.odg_last_error()


# ---------------------------------------------------------------------------------------------------- BatchedMPPI
def test_batched_plan_graph_replays_draw_fresh_noise():
    lib, L = _lib()
    from opendog_b200.mppi import BatchedMPPI
    K, S, T = 3, 64, 6
    robots = _robots(K)
    m = BatchedMPPI(robots, samples_per_robot=S, horizon=T, seed=SEED, use_graph=True)
    m.mean.copy_(torch.rand(K, T, m.A, device="cuda") - 0.5)
    rows = []
    for k in range(3):
        m.plan()
        torch.cuda.synchronize()
        rows.append(m.actions.clone())
    assert "plan" in m._graphs and int(m.iteration_dev) == 3 and m.iteration == 3
    assert not torch.equal(rows[0], rows[1]) and not torch.equal(rows[1], rows[2])
    row = torch.empty(S, m.A, device="cuda")
    for k in range(3):
        for g in range(K):
            for t in (0, T - 1):
                lib.check(L.odg_mppi_sample(p(m.mean[g, t]), 0.3, S, m.A, C.c_uint64(SEED + g), k, t, p(row), None), "sample")
                torch.cuda.synchronize()
                assert torch.equal(rows[k][t, g * S:(g + 1) * S], row), (k, g, t)
    # planning a later window of the robots
    m2 = BatchedMPPI(robots, samples_per_robot=S, horizon=T, seed=SEED, use_graph=False, num_robots=2)
    m2.mean.copy_(m.mean[1:])
    m2.plan(first_robot=1)
    # m2's group g is robot 1 + g planned with seed + g
    one = _samples(S)
    for g in range(2):
        _broadcast(one, robots, 1 + g, 1)
        a = torch.empty(T, S, m.A, device="cuda"); c = torch.empty(S, device="cuda")
        lib.check(L.odg_mppi_rollout(one._h, p(m2.mean[g]), 0.3, T, C.c_uint64(SEED + g), 0, None, 100.0, p(a), p(c), None), "rollout")
        torch.cuda.synchronize()
        assert torch.equal(m2.actions[:, g * S:(g + 1) * S], a) and torch.equal(m2.cost[g * S:(g + 1) * S], c)


def test_control_step_equals_the_loop_by_hand():
    lib, L = _lib()
    from opendog_b200.env import BatchedWalkEnv
    from opendog_b200.mppi import BatchedMPPI
    K, S, T, A, STEPS = 5, 64, 8, 8, 10

    def make_robots():
        r = BatchedWalkEnv(K, seed=7, info_keys=None)
        r.reset()
        q, v = r.get_state()
        _tilt(q, 2, 25.0)                     # robot 2 starts past the termination band: its first step ends the episode
        r.set_state(q, v)
        return r
    robots, ref_robots = make_robots(), make_robots()
    m = BatchedMPPI(robots, samples_per_robot=S, horizon=T, seed=SEED, use_graph=True)
    one = _samples(S)
    ref_mean = torch.zeros(K, T, A, device="cuda")
    ended = torch.zeros(K, dtype=torch.bool, device="cuda")
    for k in range(STEPS):
        if k == 1:
            out = m.control_step()            # the capture (synchronises before it records)
        else:
            torch.cuda.set_sync_debug_mode("error")
            try:
                out = m.control_step()
            finally:
                torch.cuda.set_sync_debug_mode("default")
        # by hand: K single-robot plans, the robots' step, the shift and the reset of ended episodes
        nm = torch.empty(K, T, A, device="cuda")
        for g in range(K):
            _broadcast(one, ref_robots, g, 1)
            a = torch.empty(T, S, A, device="cuda"); c = torch.empty(S, device="cuda")
            lib.check(L.odg_mppi_rollout(one._h, p(ref_mean[g]), 0.3, T, C.c_uint64(SEED + g), k, None, 100.0, p(a), p(c), None),
                      "rollout")
            lib.check(L.odg_mppi_reduce(p(c), p(a), T, S, A, 1.0, p(nm[g]), None, None), "reduce")
        _, rew, done, _ = ref_robots.step(nm[:, 0].contiguous())
        ref_mean[:, :-1] = nm[:, 1:]
        ref_mean[:, -1] = 0
        ref_mean[done] = 0
        torch.cuda.synchronize()
        ended |= done
        obs, reward, term, trunc = out
        q, v = robots.get_state(); rq, rv = ref_robots.get_state()
        assert torch.equal(q, rq) and torch.equal(v, rv), k
        assert torch.equal(obs, ref_robots.obs) and torch.equal(reward, ref_robots.reward), k
        assert torch.equal(term, ref_robots.terminated) and torch.equal(trunc, ref_robots.truncated), k
        assert torch.equal(m.new_mean, nm) and torch.equal(m.mean, ref_mean), k
    assert "control" in m._graphs and int(m.iteration_dev) == STEPS
    assert bool(ended[2]) and (m.mean.abs().sum() > 0)
