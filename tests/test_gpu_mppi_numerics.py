"""GPU tests of the MPPI arithmetic (include/odg_mppi.h) against independent restatements of the same operations:
the softmin reduction (`odg_mppi_reduce_groups`) bit for bit where its weights are exact and within a derived float64
bound where they are not, the sampler (`odg_mppi_sample` and the rows `odg_mppi_rollout_groups` draws) against a float64
Box-Muller restatement of the Philox stream, and the cost accumulation (`odg_mppi_accumulate`) bit for bit against
numpy float32. Non-finite sample costs (a rollout whose state went non-finite) get weight 0 and leave the group's min,
argmin and mean cost; a group with no finite cost plans a zero sequence.

Every output is the head of a guard-banded buffer (test_gpu_policy._Guarded): a sentinel tail must survive the call.

Bounds (u = 2**-24, gamma_k = k u / (1 - k u); CUDA C Programming Guide, "Mathematical Functions" appendix: expf 2 ulp,
logf 1 ulp, sincosf 2 ulp, sqrtf and float division correctly rounded; one ulp of a normal float32 y is <= 2u |y|):

* Reduce, per output element, against float64 from the kernel's own float32 inputs, x_n = (c_n - cmin) / lambda,
  w_n = exp(-x_n), W = sum w_n >= 1, N = sum w_n a_n:
  - weight: delta_n = (1 + (2 x_n + 2) u) (1 + 4u) - 1 (the argument's two roundings, then expf), plus 2**-125
    absolute for results in the subnormal range;
  - eN = sum (delta_n w_n + 2**-125) |a_n| + gamma_{S+1} sum (w_n (1 + delta_n) + 2**-125) |a_n| (products, in-order sum);
  - eW = sum delta_n w_n + S 2**-125 + gamma_{10 + ceil(S / 1024)} (W + ...) (per-thread strided sums, 10-level tree);
  - |kernel - N / W| <= (eN + |N / W| eW) / (W - eW) (1 + u) + u |N / W| (the division's rounding), plus the float64
    reference's own (S + 2) 2**-53 sum w |a| / W.
  The largest measured error / bound per shape is listed in test_reduce_general_weights_within_the_float64_bound.
* Sampler, per element, against v = mean + sigma e with e from float64 log / sqrt / cos / sin of the kernel's exact
  float32 u1, u2 and its float32-rounded argument fl(6.283185307179586f u2):
  |sigma| |e| ((1 + u)^2 (1 + 4u) (1 + u)^2 - 1) (logf's 2u halved by the sqrt, sqrtf, sincosf, the product, the
  unfused sigma * e) + u (|v| + ...) (the final add) + 2**-148 |sigma| (subnormal sin / cos).
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from test_gpu_mppi_batched import _broadcast, _robots, _samples  # noqa: E402
from test_gpu_policy import _SENTINEL, _Guarded, _cptr, _philox_np, _stream  # noqa: E402  (Philox held to the oracle there)

_SENTINEL.setdefault(torch.uint8, (torch.uint8, 0xA5))            # guard bands of u8 outputs (`alive`)

U = 2.0 ** -24
THREADS = 1024                                                    # k_mppi_reduce's block
ETA = 2.0 ** -125                                                 # absolute error of an expf result in the subnormal range
STREAM_MPPI = 0x4D505049


def _gamma(k):
    return k * U / (1 - k * U)


def _lib():
    from opendog_b200 import lib
    return lib, lib.load()


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


# ------------------------------------------------------------------------------------------------- reduce restatements
def _reduce(cost, act, G, S, lam):
    """odg_mppi_reduce_groups on float32 host arrays cost [G S], act [T][G S][A] -> (mean_out [G][T][A], stats [G][4])."""
    lib, L = _lib()
    T, N, A = act.shape
    assert N == G * S
    out, st = _Guarded((G, T, A)), _Guarded((G, 4))
    dc, da = torch.from_numpy(np.ascontiguousarray(cost)).cuda(), torch.from_numpy(np.ascontiguousarray(act)).cuda()
    lib.check(L.odg_mppi_reduce_groups(_cptr(dc), _cptr(da), T, G, S, A, lam, _cptr(out.t), _cptr(st.t), _stream()),
              "odg_mppi_reduce_groups")
    torch.cuda.synchronize()
    out.assert_tail_intact("mean_out")
    st.assert_tail_intact("stats")
    return out.t.cpu().numpy(), st.t.cpu().numpy()


def _strided_tree_sum(x):
    """k_mppi_reduce's float32 sum of x [S]: thread tid adds x[tid], x[tid + 1024], ... in order, then the fixed
    512 -> 1 tree."""
    x = np.asarray(x, np.float32)
    rows = -(-x.shape[0] // THREADS)
    pad = np.zeros(rows * THREADS, np.float32)
    pad[:x.shape[0]] = x
    s = np.zeros(THREADS, np.float32)
    for r in pad.reshape(rows, THREADS):
        s = s + r
    d = THREADS // 2
    while d:
        s[:d] = s[:d] + s[d:2 * d]
        d //= 2
    return s[0]


def _seq_sum(act, G, S, keep=None):
    """Per group, the float32 sum over samples in index order of act [T][G S][A] -> [G][T][A]; `keep` [G S] bool adds
    only those samples (a weight-0 term of the kernel's sum adds exactly 0)."""
    T, _, A = act.shape
    a = act.reshape(T, G, S, A)
    k = None if keep is None else keep.reshape(G, S)
    acc = np.zeros((T, G, A), np.float32)
    for s in range(S):
        acc = acc + (a[:, :, s] if k is None else np.where(k[None, :, s, None], a[:, :, s], np.float32(0)))
    return acc.transpose(1, 0, 2)


def _cost_mean(c):
    """stats[1]: the restated strided / tree sum of the finite costs over their count."""
    fin = np.isfinite(c)
    return np.float32(_strided_tree_sum(np.where(fin, c, np.float32(0))) / np.float32(fin.sum()))


def _softmin_bound(c, a, lam, keep=None):
    """float64 softmin of one group from the kernel's float32 inputs c [S], a [T][S][A], lam (float32 value), over the
    samples `keep` (default all), and the bound of the module docstring -> (ref [T][A], bound [T][A], W ref, W bound)."""
    c = c.astype(np.float64)
    keep = np.ones(c.shape, bool) if keep is None else keep
    S = c.shape[0]
    cmin = c[keep].min()
    x = np.where(keep, (c - cmin) / lam, np.inf)
    w = np.exp(-x)
    delta = np.where(keep, (1 + (2 * np.where(keep, x, 0) + 2) * U) * (1 + 4 * U) - 1, 0)
    aa = np.abs(a.astype(np.float64))
    W = w.sum()
    num = np.einsum("n,tna->ta", w, a.astype(np.float64))
    wa = np.einsum("n,tna->ta", w, aa)
    ref = num / W
    eN = np.einsum("n,tna->ta", delta * w + ETA, aa) + _gamma(S + 1) * np.einsum("n,tna->ta", w * (1 + delta) + ETA, aa)
    eW0 = (delta * w).sum() + S * ETA
    eW = eW0 + _gamma(10 + -(-S // THREADS)) * (W + eW0)
    q = (eN + np.abs(ref) * eW) / (W - eW)
    bound = q * (1 + U) + U * np.abs(ref) + (S + 2) * 2.0 ** -53 * wa / W
    return ref, bound, W, eW


# (G, S, T, A): every S, G, T and A value of the issue's axes, T A > 1024 (128 x 12), the planner's 1024 x 64 x 8 and
# x 12 (Go1), and 16 robots x 1024 samples
SHAPES = [(1, 1, 7, 8), (3, 2, 1, 1), (1, 1023, 7, 3), (1, 1024, 64, 8), (1, 1024, 64, 12), (3, 1025, 7, 16),
          (1, 2049, 128, 12), (3, 4097, 7, 8), (1, 12000, 64, 16), (16, 1024, 64, 8), (16, 12000, 7, 12)]
_SHAPE_IDS = [f"G{G}-S{S}-T{T}-A{A}" for G, S, T, A in SHAPES]


def _inputs(G, S, T, A, seed):
    rng = np.random.default_rng(seed)
    cost = (rng.standard_normal(G * S) * 3 + 5).astype(np.float32)
    act = rng.uniform(-1, 1, (T, G * S, A)).astype(np.float32)
    return rng, cost, act


def _boundary_positions(S):
    """Sample positions on the reduce's 1024-thread stride boundaries (and the ends), within [0, S)."""
    return sorted({p for p in (0, 1, THREADS - 1, THREADS, THREADS + 1, 2 * THREADS, S - 1) if 0 <= p < S})


@pytest.mark.parametrize("G,S,T,A", SHAPES, ids=_SHAPE_IDS)
def test_reduce_with_unit_weights_is_the_in_order_mean(G, S, T, A):
    """Equal costs (lambda 1), and random costs with ties at the minimum under lambda = 1e30: every weight is exactly
    1, so mean_out = fl(in-order float32 sum / S), stats = (min, restated strided / tree mean, S, lowest argmin)."""
    rng, cost, act = _inputs(G, S, T, A, 1)
    ref_mean = _seq_sum(act, G, S) / np.float32(S)
    equal = np.full(G * S, 3.25, np.float32)
    ties = cost.copy()
    for g in range(G):
        for p in _boundary_positions(S)[::-1][: 3 + g % 2]:
            ties[g * S + p] = np.float32(-100.0)                 # the minimum, reached at several boundary positions
    for c, lam in ((equal, 1.0), (ties, 1e30)):
        out, st = _reduce(c, act, G, S, lam)
        assert np.array_equal(_bits(out), _bits(ref_mean)), (lam, np.abs(out - ref_mean).max())
        for g in range(G):
            cg = c[g * S:(g + 1) * S]
            assert st[g, 2] == S and st[g, 0] == cg.min() and st[g, 3] == int(np.argmin(cg)), (lam, g, st[g])
            assert _bits(st[g, 1]) == _bits(_cost_mean(cg)), (lam, g, st[g, 1], _cost_mean(cg))


@pytest.mark.parametrize("G,S,T,A", SHAPES, ids=_SHAPE_IDS)
def test_reduce_with_weights_in_zero_one_is_the_subset_mean(G, S, T, A):
    """A subset at cmin, the rest at cmin + Delta with Delta / lambda >= 200 (expf underflows to exactly 0); lambda 1
    and 1e-30 (only the minima count). mean_out = the subset's in-order float32 sum over its size; argmin = its lowest
    index; stats[2] = its size."""
    rng, _, act = _inputs(G, S, T, A, 2)
    keep = np.zeros(G * S, bool)
    for g in range(G):
        pos = _boundary_positions(S)
        if S > 8:
            pos = pos + list(rng.choice(S, 5, replace=False))
        pos = pos[g % 2:] or pos                                # groups differ in their lowest member
        keep[[g * S + p for p in pos]] = True
    for lam, delta in ((1.0, 200.0), (1e-30, 1.0)):
        cost = np.where(keep, np.float32(5.0), (5.0 + delta + rng.uniform(0, 50, G * S)).astype(np.float32)).astype(np.float32)
        out, st = _reduce(cost, act, G, S, lam)
        k = keep.reshape(G, S).sum(1)
        ref = _seq_sum(act, G, S, keep) / k[:, None, None].astype(np.float32)
        assert np.array_equal(_bits(out), _bits(ref)), (lam, np.abs(out - ref).max())
        for g in range(G):
            cg = cost[g * S:(g + 1) * S]
            assert st[g, 0] == 5.0 and st[g, 2] == k[g] and st[g, 3] == int(np.argmax(keep[g * S:(g + 1) * S])), (lam, g, st[g])
            assert _bits(st[g, 1]) == _bits(_cost_mean(cg)), (lam, g)


@pytest.mark.parametrize("G,S,T,A", SHAPES, ids=_SHAPE_IDS)
def test_reduce_gives_non_finite_costs_zero_weight(G, S, T, A):
    """NaN, +inf and -inf costs on the thread-stride boundaries: mean_out and stats[0, 2, 3] equal, bit for bit, the
    same call with those costs replaced by cmin + 1e30 (weight 0 there too); stats[1] is the mean over the finite
    costs. With S = 1 the group has no finite cost: mean_out = 0, stats = (+inf, NaN, 0, -1)."""
    rng, cost, act = _inputs(G, S, T, A, 3)
    bad = np.zeros(G * S, bool)
    specials = np.array([np.nan, np.inf, -np.inf], np.float32)
    for g in range(G):
        pos = _boundary_positions(S) if S > 2 else [S - 1]
        for i, p in enumerate(pos):
            cost[g * S + p] = specials[(i + g) % 3]
            bad[g * S + p] = True
    out, st = _reduce(cost, act, G, S, 0.7)
    if S == 1:
        assert not out.any() and not np.signbit(out).any()
        assert (st[:, 0] == np.inf).all() and np.isnan(st[:, 1]).all() and (st[:, 2] == 0).all() and (st[:, 3] == -1).all()
        return
    repl = cost.copy()
    for g in range(G):
        sl = slice(g * S, (g + 1) * S)
        repl[sl] = np.where(bad[sl], np.float32(cost[sl][~bad[sl]].min() + np.float32(1e30)), cost[sl])
    rout, rst = _reduce(repl, act, G, S, 0.7)
    assert np.isfinite(out).all() and np.array_equal(_bits(out), _bits(rout))
    assert np.array_equal(_bits(st[:, [0, 2, 3]]), _bits(rst[:, [0, 2, 3]]))
    for g in range(G):
        assert _bits(st[g, 1]) == _bits(_cost_mean(cost[g * S:(g + 1) * S])), g


@pytest.mark.parametrize("S", [1, 1025, 12000])
def test_reduce_group_without_a_finite_cost_plans_zero(S):
    """Group 1 of 3 has only NaN / +-inf costs: mean_out[1] = +0, stats[1] = (+inf, NaN, 0, -1); groups 0 and 2 are
    bit-identical to the call in which group 1's costs are finite."""
    G, T, A = 3, 7, 12
    rng, cost, act = _inputs(G, S, T, A, 4)
    finite = cost.copy()
    cost[S:2 * S] = np.array([np.nan, np.inf, -np.inf], np.float32)[np.arange(S) % 3]
    out, st = _reduce(cost, act, G, S, 1.0)
    fout, fst = _reduce(finite, act, G, S, 1.0)
    assert not out[1].any() and not np.signbit(out[1]).any()
    assert st[1, 0] == np.inf and np.isnan(st[1, 1]) and st[1, 2] == 0 and st[1, 3] == -1
    for g in (0, 2):
        assert np.array_equal(_bits(out[g]), _bits(fout[g])) and np.array_equal(_bits(st[g]), _bits(fst[g])), g


@pytest.mark.parametrize("G,S,T,A", SHAPES, ids=_SHAPE_IDS)
def test_reduce_general_weights_within_the_float64_bound(G, S, T, A):
    """Costs 1e4 + spread U(0, 1) for spreads 0.1, 10 and 200 lambda and lambda in {1e-3, 1, 1e3} (c - cmin rounds),
    against float64 from the same float32 inputs at the module docstring's bound. stats[0, 3] exact, stats[1] the
    restated mean bit for bit, stats[2] within its own bound.

    Largest measured error / bound over the nine cases, on an NVIDIA B200 (1000 W power limit), per (G, S, T, A):
    (1, 1, 7, 8) 0 (one sample: the mean is that sample's row); (3, 2, 1, 1) 0.040; (1, 1023, 7, 3) 0.0035;
    (1, 1024, 64, 8) 0.0085; (1, 1024, 64, 12) 0.0071; (3, 1025, 7, 16) 0.0057; (1, 2049, 128, 12) 0.0039;
    (3, 4097, 7, 8) 0.0012; (1, 12000, 64, 16) 0.00067; (16, 1024, 64, 8) 0.0077; (16, 12000, 7, 12) 0.00050.
    The bound is a worst case over rounding signs; in-order sums of random-sign terms stay far below it."""
    rng, _, act = _inputs(G, S, T, A, 5)
    worst = 0.0
    for lam in (1e-3, 1.0, 1e3):
        lam32 = float(np.float32(lam))
        for spread in (0.1, 10.0, 200.0):
            cost = (1e4 + spread * lam * rng.uniform(0, 1, G * S)).astype(np.float32)
            out, st = _reduce(cost, act, G, S, lam)
            for g in range(G):
                sl = slice(g * S, (g + 1) * S)
                cg = cost[sl]
                ref, bound, W, eW = _softmin_bound(cg, act[:, sl], lam32)
                err = np.abs(out[g].astype(np.float64) - ref)
                assert (err <= bound).all(), (lam, spread, g, float((err / bound).max()))
                worst = max(worst, float((err / bound).max()))
                assert st[g, 0] == cg.min() and st[g, 3] == int(np.argmin(cg)), (lam, spread, g)
                assert _bits(st[g, 1]) == _bits(_cost_mean(cg)) and abs(float(st[g, 2]) - W) <= eW, (lam, spread, g)
    print(f"\nreduce error / bound G{G} S{S} T{T} A{A}: {worst:.3g}")


# ------------------------------------------------------------------------------------------------- sampler
def _sample_ref(mean, sigma, rows, A, seed, iteration, t):
    """float64 restatement of odg_core.cuh mppi_sample_row for sample ids `rows` -> (v = mean + sigma eps unclamped
    [n][A], bound [n][A]). u1, u2 and the float32 argument of sincosf are the kernel's exact values."""
    eps = []
    for blk in range((A + 3) // 4):
        r = _philox_np(seed, np.asarray(rows, np.uint64), iteration, ((t << 8) | blk) & 0xFFFFFFFF, STREAM_MPPI)
        for pr in range(2):
            u1 = ((r[2 * pr] >> 8).astype(np.float64) + 1.0) * 2.0 ** -24         # exact in float32 too
            u2 = (r[2 * pr + 1] >> 8).astype(np.float64) * 2.0 ** -24
            arg = (np.float32(6.283185307179586) * u2.astype(np.float32)).astype(np.float64)
            rad = np.sqrt(-2.0 * np.log(u1))
            eps += [rad * np.cos(arg), rad * np.sin(arg)]
    e = np.stack(eps[:A], axis=1)
    m, s = np.asarray(mean, np.float64)[None, :], float(np.float32(sigma))
    v = m + s * e
    se = np.abs(s * e)
    rel = (1 + U) ** 2 * (1 + 4 * U) * (1 + U) ** 2 - 1
    bound = se * rel + U * (np.abs(v) + se * rel) + 2.0 ** -148 * abs(s)
    return v, bound


def _check_rows(got, mean, sigma, rows, A, seed, iteration, t, what):
    v, bound = _sample_ref(mean, sigma, rows, A, seed, iteration, t)
    clipped = np.clip(v, -1.0, 1.0)
    err = np.abs(got.astype(np.float64) - clipped)
    assert (err <= bound).all(), (what, float((err / np.maximum(bound, 1e-300)).max()))
    far = np.abs(v) > 1.0 + bound
    assert (got[far] == np.sign(v[far])).all(), what                   # beyond the clamp by more than the bound: exactly +-1


_SEEDS = (0, 2 ** 32 - 1, 2 ** 32, 2 ** 64 - 1)
_NS = (1, 127, 128, 129, 12000)
_TS = (0, 255, 256, 65535)
_ITS = (0, 2 ** 31, 2 ** 32 - 1)
_MEAN16 = np.array([-1.0, 1.0, -0.99, 0.995, -1.5, 1.5, 0.0, 0.3, -0.7, 1 - 2 ** -24, -(1 - 2 ** -24), 0.5, -0.05, 2.0,
                    -2.0, 0.9], np.float32)


@pytest.mark.parametrize("A", range(1, 17))
def test_sample_matches_the_box_muller_restatement(A):
    """Every element of odg_mppi_sample for act_dim A (1-4 Philox blocks), with N, t, iteration and the 64-bit seed
    rotating through their edge values, sigma in {0, 0.3, 5} and nominal entries at and beyond +-1. sigma = 0 gives
    exactly clamp(mean)."""
    lib, L = _lib()
    N, t, it, seed = _NS[A % 5], _TS[A % 4], _ITS[A % 3], _SEEDS[(A // 4) % 4]
    mean = np.roll(_MEAN16, A)[:A].copy()
    dm = torch.from_numpy(mean).cuda()
    for sigma in (0.0, 0.3, 5.0):
        act = _Guarded((N, A))
        lib.check(L.odg_mppi_sample(_cptr(dm), sigma, N, A, C.c_uint64(seed), it, t, _cptr(act.t), _stream()), "sample")
        torch.cuda.synchronize()
        act.assert_tail_intact("action")
        got = act.t.cpu().numpy()
        if sigma == 0.0:
            assert np.array_equal(got, np.broadcast_to(np.clip(mean, -1, 1), got.shape)), (A, N)
        else:
            _check_rows(got, mean, sigma, np.arange(N), A, seed, it, t, (A, N, t, it, seed, sigma))


def test_rollout_groups_rows_match_the_restatement_go1():
    """The action rows odg_mppi_rollout_groups writes on Go1 (A = 12, three Philox blocks): G = 3, S = 37, seed
    2**32 - 2 (seed + g carries into the high word) and a device plan counter preset to 2**31 + 3. Row (t, g S + s) is
    the restatement with key seed + g, sample s, that counter and mean[g][t]."""
    lib, L = _lib()
    G, S, T, seed, it = 3, 37, 10, 2 ** 32 - 2, 2 ** 31 + 3
    robots = _robots(G, model="go1", tilt=1, auto_reset=0)
    smp = _samples(G * S, model="go1")
    A = smp.act_dim
    assert A == 12
    _broadcast(smp, robots, 0, G)
    rng = np.random.default_rng(6)
    mean = rng.uniform(-1.2, 1.2, (G, T, A)).astype(np.float32)
    dm = torch.from_numpy(mean).cuda()
    it_dev = torch.from_numpy(np.array([it], np.uint32).view(np.int32)).cuda()
    acts, cost = _Guarded((T, G * S, A)), _Guarded((G * S,))
    lib.check(L.odg_mppi_rollout_groups(smp._h, G, _cptr(dm), 0.3, T, C.c_uint64(seed), 0, _cptr(it_dev), 100.0,
                                        _cptr(acts.t), _cptr(cost.t), _stream()), "odg_mppi_rollout_groups")
    torch.cuda.synchronize()
    acts.assert_tail_intact("actions")
    cost.assert_tail_intact("cost")
    got = acts.t.cpu().numpy()
    assert np.isfinite(cost.t.cpu().numpy()).all()
    for g in range(G):
        for t in range(T):
            _check_rows(got[t, g * S:(g + 1) * S], mean[g, t], 0.3, np.arange(S), A, seed + g, it, t, (g, t))


# ------------------------------------------------------------------------------------------------- accumulate
@pytest.mark.parametrize("N", [1, 255, 256, 257, 100003])
@pytest.mark.parametrize("term_cost", [0.0, 100.0])
def test_accumulate_matches_float32_restatement(N, term_cost):
    """Five chained odg_mppi_accumulate calls, bit for bit against numpy float32: rewards with +-0, subnormals and
    +-1e30, samples dead from the start (alive 0) and alive flags other than 1; dead samples' cost and alive are
    untouched."""
    lib, L = _lib()
    rng = np.random.default_rng(N + int(term_cost))
    specials = np.array([0.0, -0.0, 1e-40, -1e-40, 1.4e-45, -1.4e-45, 1e30, -1e30, 3.0e38], np.float32)

    def values(n):
        x = (rng.standard_normal(n) * 4).astype(np.float32)
        pick = rng.random(n) < 0.3
        x[pick] = specials[rng.integers(0, len(specials), int(pick.sum()))]
        return x
    cost0 = values(N)
    alive0 = rng.choice(np.array([0, 1, 1, 1, 255], np.uint8), N)
    cost, alive = _Guarded((N,)), _Guarded((N,), dtype=torch.uint8)
    cost.t.copy_(torch.from_numpy(cost0))
    alive.t.copy_(torch.from_numpy(alive0))
    c, al = cost0.copy(), alive0.copy()
    for _ in range(5):
        rew = values(N)
        term = (rng.random(N) < 0.15).astype(np.uint8)
        dr, dt = torch.from_numpy(rew).cuda(), torch.from_numpy(term).cuda()
        lib.check(L.odg_mppi_accumulate(_cptr(dr), _cptr(dt), N, term_cost, _cptr(cost.t), _cptr(alive.t), _stream()),
                  "odg_mppi_accumulate")
        live = al != 0
        with np.errstate(over="ignore"):
            step = c - rew
            step = np.where(term != 0, step + np.float32(term_cost), step)
        c = np.where(live, step, c).astype(np.float32)
        al = np.where(live & (term != 0), np.uint8(0), al).astype(np.uint8)
    torch.cuda.synchronize()
    cost.assert_tail_intact("cost")
    alive.assert_tail_intact("alive")
    assert np.array_equal(_bits(cost.t.cpu().numpy()), _bits(c))
    assert np.array_equal(alive.t.cpu().numpy(), al)
    dead = alive0 == 0
    assert np.array_equal(_bits(cost.t.cpu().numpy()[dead]), _bits(cost0[dead]))


# ------------------------------------------------------------------------------------------------- the step-by-step loop
def test_step_by_step_loop_equals_the_fused_rollout():
    """The loop include/odg_mppi.h documents — odg_mppi_sample -> BatchedWalkEnv.step (reward_unclipped, terminated)
    -> odg_mppi_accumulate, T = 10, N = 128 — equals odg_mppi_rollout's action rows and costs bit for bit. Half the
    samples start from a landed robot, half from the same robot tilted past the termination band."""
    lib, L = _lib()
    from opendog_b200.env import BatchedWalkEnv
    N, T, sigma, seed, it = 128, 10, 0.3, 2 ** 32 - 2, 7
    robots = _robots(2, tilt=1, auto_reset=0)
    fused = _samples(N)
    stepped = BatchedWalkEnv(N, seed=11, info_keys=("reward_unclipped",), auto_reset=0)
    _broadcast(fused, robots, 0, 2)
    _broadcast(stepped, robots, 0, 2)
    A = fused.act_dim
    mean = (torch.rand(T, A, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8)) - 0.5).contiguous()
    ref_a, ref_c = _Guarded((T, N, A)), _Guarded((N,))
    lib.check(L.odg_mppi_rollout(fused._h, _cptr(mean), sigma, T, C.c_uint64(seed), it, None, 100.0, _cptr(ref_a.t),
                                 _cptr(ref_c.t), _stream()), "odg_mppi_rollout")
    cost, alive = _Guarded((N,)), _Guarded((N,), dtype=torch.uint8)
    cost.t.zero_()
    alive.t.fill_(1)
    rows = _Guarded((T, N, A))
    for t in range(T):
        lib.check(L.odg_mppi_sample(_cptr(mean[t]), sigma, N, A, C.c_uint64(seed), it, t, _cptr(rows.t[t]), _stream()), "sample")
        stepped.step(rows.t[t])
        lib.check(L.odg_mppi_accumulate(_cptr(stepped.info["reward_unclipped"]), _cptr(stepped.terminated), N, 100.0,
                                        _cptr(cost.t), _cptr(alive.t), _stream()), "odg_mppi_accumulate")
    torch.cuda.synchronize()
    for g in (ref_a, ref_c, cost, alive, rows):
        g.assert_tail_intact("loop output")
    assert torch.equal(rows.t, ref_a.t)
    assert torch.equal(cost.t.view(torch.int32), ref_c.t.view(torch.int32))
    n_alive = int(alive.t.sum())
    assert 0 < n_alive < N and bool((alive.t[N // 2:] == 0).all())      # the tilted half terminated, paying 100 once
    assert bool((cost.t[N // 2:] > 50).all())


# ------------------------------------------------------------------------------------------------- end to end
def test_non_finite_samples_get_zero_weight_end_to_end():
    """Three robots broadcast into 3 x 256 samples; two samples of group 1 get a NaN qvel (get_state / set_state; the
    control handle takes the same round trip unmodified, since set_state restarts the warm start). After
    odg_mppi_rollout_groups + odg_mppi_reduce_groups on both: groups 0 and 2 are bit-identical, group 1's two costs are
    non-finite, and its new mean is finite, equal to the reduce of its costs with those two replaced by cmin + 1e30,
    and within the float64 bound of the softmin over its other 254 samples."""
    lib, L = _lib()
    K, S, T, lam, seed = 3, 256, 8, 1.0, 2 ** 32 - 2
    robots = _robots(K, auto_reset=0)
    hs = [_samples(K * S), _samples(K * S)]
    bad = [S + 5, S + 200]
    for i, h in enumerate(hs):
        _broadcast(h, robots, 0, K)
        q, v = h.get_state()
        torch.cuda.synchronize()
        if i == 0:
            v[bad[0], 0] = float("nan")
            v[bad[1], 3] = float("nan")
        h.set_state(q, v)
    A = hs[0].act_dim
    mean = (torch.rand(K, T, A, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9)) - 0.5).contiguous()
    res = []
    for h in hs:
        a, c = _Guarded((T, K * S, A)), _Guarded((K * S,))
        nm, st = _Guarded((K, T, A)), _Guarded((K, 4))
        lib.check(L.odg_mppi_rollout_groups(h._h, K, _cptr(mean), 0.3, T, C.c_uint64(seed), 0, None, 100.0, _cptr(a.t), _cptr(c.t),
                                            _stream()), "odg_mppi_rollout_groups")
        lib.check(L.odg_mppi_reduce_groups(_cptr(c.t), _cptr(a.t), T, K, S, A, lam, _cptr(nm.t), _cptr(st.t), _stream()),
                  "odg_mppi_reduce_groups")
        torch.cuda.synchronize()
        for gb in (a, c, nm, st):
            gb.assert_tail_intact("plan output")
        res.append([x.t.cpu().numpy() for x in (a, c, nm, st)])
    (a, c, nm, st), (ca, cc, cnm, cst) = res
    for g in (0, 2):
        sl = slice(g * S, (g + 1) * S)
        assert np.array_equal(_bits(a[:, sl]), _bits(ca[:, sl])) and np.array_equal(_bits(c[sl]), _bits(cc[sl])), g
        assert np.array_equal(_bits(nm[g]), _bits(cnm[g])) and np.array_equal(_bits(st[g]), _bits(cst[g])), g
    c1, a1 = c[S:2 * S].copy(), np.ascontiguousarray(a[:, S:2 * S])
    nonfin = ~np.isfinite(c1)
    assert sorted(np.flatnonzero(nonfin) + S) == bad
    assert np.isfinite(nm[1]).all() and np.isfinite(st[1, :3]).all()
    repl = np.where(nonfin, np.float32(c1[~nonfin].min() + np.float32(1e30)), c1).astype(np.float32)
    rout, rst = _reduce(repl, a1, 1, S, lam)
    assert np.array_equal(_bits(nm[1]), _bits(rout[0])) and np.array_equal(_bits(st[1, [0, 2, 3]]), _bits(rst[0, [0, 2, 3]]))
    assert _bits(st[1, 1]) == _bits(_cost_mean(c1))
    ref, bound, _, _ = _softmin_bound(c1, a1, float(np.float32(lam)), keep=~nonfin)
    assert (np.abs(nm[1].astype(np.float64) - ref) <= bound).all()
