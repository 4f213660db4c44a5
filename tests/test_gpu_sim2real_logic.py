"""The QuadrupedEnv post-physics logic (`k_s2r_pre`, `k_s2r_post`, `k_s2r_reset` of odg_sim2real.cu) against the
reference's own post-physics code (oracle/sim2real_oracle.py) on IDENTICAL post-physics states, for both trainers
(train: 22 obs / 4 actions, terrain: 12 obs / 8 actions) at N in {1, 127, 128, 129, 4097}: one env, exactly one 128-env
block, one block plus one env, many blocks with a state stride (N rounded up to 64) that differs from N.

Harness: the GPU env steps with auto_reset = 0; its post-physics state (`get_state`) is copied into an oracle whose
`sim.step` is a no-op, with `counter`, `prev_x`, cumulative sums, `prev_net` and `last_cmd` set to what the GPU was given
through `set_bookkeeping`. Later steps chain: the oracle carries its own bookkeeping, so the kernel's write-back is
checked too. Every output is the head of a buffer whose tail holds a sentinel (NaN payload / 0xAB) that must survive.

Tolerances, derived from what differs between the two sides:
* sim_target_rad: float32(oracle cmd), bit for bit (a clip of home + a * amp in double, rounded once).
* obs: joint positions / velocities, v_x and the phase entries bit-exact; yaw / pitch / roll bit-exact or one float32
  ulp (device atan2 / asin against host libm may differ in the last double bit). For a non-finite quaternion both
  sides take pitch = copysign(pi / 2, NaN): the NaN's sign bit is not specified, so there |pitch| is compared.
* reward: one float32 ulp of the oracle's reward, plus the smoothness term's bound from rounded targets: the kernel
  squares float32(cmd) - float32(last_cmd), the reference cmd - last_cmd in double; with e_k = |float32(cmd_k) - cmd_k|
  + |float32(last_k) - last_k| and d_k = cmd_k - last_k the term differs by at most c * sum(2 |d_k| e_k + e_k^2)
  (c = 0.01 train, 0.005 terrain), computed per env; plus 1e-11 for the two double evaluations of a sum of terms
  below 1e4. Non-finite rewards must be equal (NaN with NaN).
* done / reason: bit-exact on every env.
* leg deviation (train): dev = |deg(cmd - home)| is compared with 15 and 40 from the float32 target. Where the oracle's
  dev lies within 57.3 * e_k (+ 4 ulp(128) for the kernel's real_home_deg round trip) of a threshold the kernel may
  decide the other way; such a flip moves the reward by a multiple of 0.5 and is accepted only there. With this model's
  ctrlrange no target is more than 25.4 degrees from home, so the 40-degree `too_far` rule cannot fire (asserted).

Branch cases (set_state, which zeroes the solver warm start, then a two-pass replay: step, read x', set the same
pre-state again, check the post-state repeats bit for bit, and choose the bookkeeping from x' in double): dx = 0,
+-1e-9, +-1e-3; dnet at 0.0005 and one double ulp to either side; cpos at 0.05 +- ulp; cneg at and one ulp past
0.75 * cpos (train) / 0.85 * cpos (terrain); backward trunk velocities around -0.005; roll / pitch / yaw on both sides
of 5 / 10 / 25 degrees (train) and 15 / 35 / 35 / 52.5 (terrain), yaw-only 45 degrees among them; trunk heights on
both sides of settled_z - 0.03 and init_z +- 0.05; actions in [-2, 2] (ctrlrange clipping) and placed inside and just
outside the rounding margin of the 15-degree rule in both counter parities; NaN / +-inf injected into qpos / qvel,
alone and with the trunk rolled past the orientation limit. The physics keeps the quaternion of such a state finite, so
with the tilt the orientation rule and mj_error coincide: the train variant (no `not done` guard in the reference)
reports orientation_limit with both penalties, the terrain variant keeps mj_error; both outcomes are asserted reached.

Episode ends with auto_reset: the max_steps cap (250 / the terrain default 1000) ends an episode with reason
max_steps and no penalty, a termination on the same step wins, terminal_obs is the oracle's obs, the returned obs is
the settled reset obs, and the next step is a fresh episode (counter 0, prev_x = settled x, zero sums, last_cmd =
float32 home ctrl), checked against an oracle given exactly that bookkeeping; the same for termination-driven resets.
Masked reset: masked envs get the settled state, fresh bookkeeping and their obs row; the others keep all of it.

Terrain fields (odg_terrain.cu): an environment's field is drawn from Philox4x32-10 keyed by (seed; global env id =
first_env_id + env, the env's generation counter, cell pair or 0xFFFFFFFF, stream "TERR"), and the generation counter
advances by one per regeneration. So the flat / rough choice of every (env, generation) is predictable from the first
word of the 0xFFFFFFFF draw (flat iff < 2^31); a regenerated field differs from its predecessor unless both draws are
flat; and two shards with first_env_id 0 / n0 reproduce the N-env batch's fields after the same masked resets.

At N = 4097 the oracle checks a fixed seeded sample: the first and last env of every 128-env block, the first 160
envs (every case) and 384 more; the sentinels and the whole-batch assertions cover every env.
"""
import ctypes as C
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from test_gpu_policy import _philox_np  # noqa: E402  (held to the oracle's Philox by a CPU test there)

NS = (1, 127, 128, 129, 4097)
VARIANTS = ("train", "terrain")
REASON = {"max_steps": 0, "mj_error": 1, "orientation_limit": 2, "too_much_backward": 3}
SMOOTH_C = {"train": 0.01, "terrain": 0.005}
BACK_F = {"train": 0.75, "terrain": 0.85}
MAX_STEPS = {"train": 250, "terrain": 1000}
DEG = 57.29577951308232
DEG_SLACK = 4 * float(np.spacing(128.0))
DOUBLE_SLACK = 1e-11
F_SENT, B_SENT, TAIL = 0x7FA1B2C3, 0xAB, 64


def _cptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class _Buf:
    """An output at the head of a longer device buffer whose tail (and, after `fill`, whole body) holds a sentinel."""

    def __init__(self, shape, dtype=torch.float32):
        self.n = math.prod(shape)
        self.buf = torch.empty(self.n + TAIL, dtype=dtype, device="cuda")
        self.t = self.buf[:self.n].view(shape)
        self.fill()

    def fill(self):
        if self.buf.dtype == torch.float32:
            self.buf.view(torch.int32).fill_(F_SENT)
        else:
            self.buf.fill_(B_SENT)

    def is_sentinel(self):
        if self.buf.dtype == torch.float32:
            return (self.buf.view(torch.int32) == F_SENT)[:self.n].view(self.t.shape).cpu().numpy()
        return (self.buf == B_SENT)[:self.n].view(self.t.shape).cpu().numpy()

    def assert_tail(self, what):
        tail = self.buf[self.n:]
        bad = int((tail.view(torch.int32) != F_SENT).sum()) if tail.dtype == torch.float32 else int((tail != B_SENT).sum())
        assert bad == 0, f"{what}: {bad} elements written past the end of the output"


class _Env:
    """A BatchedQuadrupedEnv driven through the C ABI with guarded outputs."""

    def __init__(self, variant, N, auto_reset=False, max_steps=None):
        from opendog_b200 import lib
        from opendog_b200.compat import BatchedQuadrupedEnv
        self.lib, self.L = lib, lib.load()
        self.e = BatchedQuadrupedEnv(N, variant=variant, auto_reset=auto_reset, max_steps=max_steps)
        self.N, self.od, self.ad = N, self.e.obs_dim, self.e.act_dim
        self.out = {"obs": _Buf((N, self.od)), "reward": _Buf((N,)), "done": _Buf((N,), torch.uint8),
                    "reason": _Buf((N,), torch.uint8), "target": _Buf((N, 8)), "tobs": _Buf((N, self.od))}

    def step(self, a):
        a = torch.as_tensor(np.asarray(a, np.float32)).to("cuda").contiguous()
        o = self.out
        self.lib.check(self.L.odg_s2r_step(self.e._h, _cptr(a), _cptr(o["obs"].t), _cptr(o["reward"].t), _cptr(o["done"].t),
                                           _cptr(o["reason"].t), _cptr(o["target"].t), _cptr(o["tobs"].t), self.e._stream()),
                       "odg_s2r_step")
        torch.cuda.synchronize()
        for k, b in o.items():
            b.assert_tail(k)
        return {k: b.t.cpu().numpy().copy() for k, b in o.items()}

    def reset(self, mask=None):
        m = None if mask is None else torch.as_tensor(np.asarray(mask, np.uint8)).to("cuda").contiguous()
        self.out["obs"].fill()
        self.lib.check(self.L.odg_s2r_reset(self.e._h, _cptr(m), _cptr(self.out["obs"].t), self.e._stream()), "odg_s2r_reset")
        torch.cuda.synchronize()
        self.out["obs"].assert_tail("reset obs")
        return self.out["obs"].t.cpu().numpy().copy()

    def state(self):
        q, v = self.e.sim.get_state()
        return q.cpu().numpy().copy(), v.cpu().numpy().copy()

    def set_state(self, q, v):
        self.e.sim.set_state(torch.from_numpy(np.ascontiguousarray(q, np.float32)), torch.from_numpy(np.ascontiguousarray(v, np.float32)))

    def set_bk(self, bk):
        self.e.set_bookkeeping(counter=torch.from_numpy(bk["counter"].astype(np.int32)), prev_x=torch.from_numpy(bk["prev_x"]),
                               cum_pos=torch.from_numpy(bk["cpos"]), cum_neg=torch.from_numpy(bk["cneg"]),
                               prev_net=torch.from_numpy(bk["prev_net"]),
                               last_cmd=torch.from_numpy(bk["last_cmd"].astype(np.float32)))


class _Ref:
    """One oracle instance with a no-op physics step: only the reference's post-physics code runs."""

    def __init__(self, variant, settled_z):
        from oracle.sim2real_oracle import QuadrupedEnvOracle, QuadrupedEnvV2Oracle
        self.variant = variant
        self.o = QuadrupedEnvOracle() if variant == "train" else QuadrupedEnvV2Oracle(terrain=False)
        self.o.sim.step = lambda: None
        self.o.n_sub = 1                           # one no-op substep: min_gap is not used here
        if variant == "terrain":
            self.o.settled_z = float(settled_z)     # current_initial_body_z_pos: the GPU's settled trunk height
        self.cattr = "counter" if variant == "train" else "steps"
        self.act_id = list(self.o.act_id)
        self.home = np.array(self.o.home)
        self.home_ctrl32 = np.array(self.o.initial_ctrl, np.float32)

    def step(self, q, v, bk, i, a):
        o = self.o
        o.sim.qpos[:] = q; o.sim.qvel[:] = v
        setattr(o, self.cattr, int(bk["counter"][i]))
        o.prev_x, o.cpos, o.cneg, o.prev_net = (float(bk[k][i]) for k in ("prev_x", "cpos", "cneg", "prev_net"))
        o.last_cmd = np.array(bk["last_cmd"][i], np.float64)
        obs, r, done, info = o.step(a)
        new = dict(counter=getattr(o, self.cattr), prev_x=o.prev_x, cpos=o.cpos, cneg=o.cneg, prev_net=o.prev_net,
                   last_cmd=np.array(o.last_cmd, np.float64))
        return obs, r, done, REASON[info["termination_reason"]], np.asarray(info["sim_target_rad"], np.float64), new


def _bk_new(N):
    return dict(counter=np.zeros(N, np.int64), prev_x=np.zeros(N), cpos=np.zeros(N), cneg=np.zeros(N), prev_net=np.zeros(N),
                last_cmd=np.zeros((N, 8)))


def _bk_set_row(bk, i, row):
    for k, v in row.items():
        bk[k][i] = v


def _sample(N, extra=384):
    if N <= 160:
        return np.arange(N)
    edges = [e for b in range(0, N, 128) for e in (b, min(b + 127, N - 1))]
    rng = np.random.default_rng(4097)
    return np.unique(np.concatenate([edges, np.arange(160), rng.choice(N, extra, replace=False)]))


def _ulp_close(g, r):
    """g equals r or is its float32 neighbour."""
    r = np.float32(r)
    return g == r or g == np.nextafter(r, np.float32(np.inf)) or g == np.nextafter(r, np.float32(-np.inf))


class _Stats(dict):
    def __missing__(self, k):
        return 0

    def counts(self):
        return {k: v for k, v in self.items() if not isinstance(v, list)}


def _check_obs(g, r, quat_finite, what, st):
    assert np.array_equal(g[3:], r[3:], equal_nan=True), f"{what}: joint / velocity / phase entries {g[3:]} vs {r[3:]}"
    for k in range(3):
        if np.array_equal(g[k:k + 1], r[k:k + 1], equal_nan=True):
            continue
        if np.isfinite(r[k]) and np.isfinite(g[k]) and _ulp_close(g[k], r[k]):
            st["ypr_ulp"] += 1
            continue
        if k == 1 and not quat_finite and abs(g[k]) == abs(r[k]) == np.float32(math.pi / 2):
            st["nan_pitch_sign"] += 1
            continue
        raise AssertionError(f"{what}: ypr[{k}] {g[k]!r} vs {r[k]!r}")


def _leg_penalties(devs, margins, phase):
    """The train variant's leg rule (train.py:340-383) for every way the comparisons within their rounding margin of a
    threshold may go: the set of possible penalties, and the number of such comparisons."""
    amb, fixed = [], {}
    for k in range(8):
        for thr in (15.0, 40.0):
            if abs(devs[k] - thr) <= margins[k]:
                amb.append((k, thr))
            else:
                fixed[(k, thr)] = devs[k] > thr
    out = set()
    for m in range(1 << len(amb)):
        dec = dict(fixed)
        for b, key in enumerate(amb):
            dec[key] = bool(m >> b & 1)
        tf = nh = 0
        for leg in range(4):
            swinging = (leg in (0, 3)) if phase == 0 else (leg in (1, 2))
            if swinging:
                tf += any(dec[(leg * 2 + j, 40.0)] for j in range(2))
            else:
                nh += any(dec[(leg * 2 + j, 15.0)] for j in range(2))
        out.add((tf + nh) * 0.5)
    return out, len(amb)


def _check_reward(variant, rk, ro, cmd, last_or, last_gpu, ref, phase, what, st):
    if not (np.isfinite(rk) and np.isfinite(ro)):
        assert np.array_equal(np.float32([rk]), np.float32([ro]), equal_nan=True), f"{what}: reward {rk!r} vs {ro!r}"
        return
    cmd32 = cmd.astype(np.float32).astype(np.float64)
    e = np.abs(cmd32 - cmd) + np.abs(last_gpu - last_or)
    d = np.abs(cmd - last_or)
    bound = SMOOTH_C[variant] * float(np.sum(2 * d * e + e * e)) + DOUBLE_SLACK
    alts, p_or = {0.0}, 0.0
    if variant == "train":
        devs = np.array([abs(math.degrees(cmd[ref.act_id[k]] - ref.home[k])) for k in range(8)])
        margins = DEG * np.abs(cmd32 - cmd)[ref.act_id] * (1 + 1e-12) + DEG_SLACK
        alts, namb = _leg_penalties(devs, margins, phase)
        p_or = _leg_penalties(devs, np.full(8, -1.0), phase)[0].pop()
        st["margin_inside"] += namb
        for k in range(8):
            if margins[k] < abs(devs[k] - 15.0) <= 4 * margins[k]:
                st["margin_just_outside"] += 1
    for p in sorted(alts, key=lambda p: abs(p - p_or)):
        want = ro + p_or - p
        tol = float(np.spacing(np.float32(abs(want)))) + bound
        if abs(float(rk) - want) <= tol:
            if p != p_or:
                st["leg_flips"] += 1
            return
    raise AssertionError(f"{what}: reward {rk!r} vs oracle {ro!r} (bound {bound:.3e}, leg penalties {sorted(alts)}, oracle {p_or})")


def _check_step(variant, ref, out, q, v, bk, last_gpu, a, idx, what, st, expect_done=None, reset_obs=None):
    """Compare the GPU step outputs `out` of envs `idx` with the oracle on post-physics state (q, v) and bookkeeping
    `bk` (updated in place with the oracle's write-back; `last_gpu` with the GPU's float32 targets)."""
    from oracle.sim2real_oracle import quat_to_ypr
    for i in idx:
        w = f"{what} env {i}"
        last_or = bk["last_cmd"][i].copy()
        phase = int(bk["counter"][i]) % 2
        ro, rr, rd, rreason, cmd, new = ref.step(q[i].astype(np.float64), v[i].astype(np.float64), bk, i, a[i])
        assert np.array_equal(out["target"][i], cmd.astype(np.float32)), f"{w}: sim_target_rad"
        qf = bool(np.isfinite(q[i, 3:7]).all())
        _check_obs(out["tobs"][i], ro, qf, w + " terminal_obs", st)
        done = rd if expect_done is None else (rd or bool(expect_done[i]))
        assert out["done"][i] == done and out["reason"][i] == rreason, f"{w}: done/reason {out['done'][i]}/{out['reason'][i]} vs {done}/{rreason}"
        if done and reset_obs is not None:
            assert np.array_equal(out["obs"][i], reset_obs), f"{w}: returned obs is not the settled reset obs"
        else:
            _check_obs(out["obs"][i], ro, qf, w + " obs", st)
        _check_reward(variant, float(out["reward"][i]), rr, cmd, last_or, last_gpu[i], ref, phase, w, st)
        st["checked"] += 1
        st[f"reason{rreason}"] += 1
        if np.isfinite(q[i, 3:7]).all():
            y, p, r = quat_to_ypr(q[i, 3:7].astype(np.float64))
            if not (np.isfinite(q[i]).all() and np.isfinite(v[i]).all()):
                lim = math.radians(25.0 if variant == "train" else 35.0)
                st["mj_error_with_orientation"] += abs(r) > lim or abs(p) > lim or abs(y) > lim * (1.0 if variant == "train" else 1.5)
            else:
                st.setdefault("ang", []).append((abs(r), abs(p), abs(y)))
                st.setdefault("z", []).append(float(q[i, 2]))
                st.setdefault("vx", []).append(float(v[i, 0]))
        _bk_set_row(bk, i, new)
        last_gpu[i] = out["target"][i].astype(np.float64)


def _same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a, np.float32).view(np.int32), np.ascontiguousarray(b, np.float32).view(np.int32))


def _quat(axis, deg):
    h = math.radians(deg) / 2
    q = [math.cos(h), 0.0, 0.0, 0.0]
    q[1 + axis] = math.sin(h)
    return q


def _cases(variant):
    """(name, spec) of every branch case; spec keys: bk (bookkeeping rule from x'), q/v (pre-state edits), a (action)."""
    f = BACK_F[variant]
    up, dn = (lambda x: np.nextafter(x, np.inf)), (lambda x: np.nextafter(x, -np.inf))
    cs = []
    for dx in (0.0, 1e-9, -1e-9, 1e-3, -1e-3):
        cs.append((f"dx={dx}", dict(bk=dict(dx=dx, cpos=0.03, cneg=0.01, prev_net=0.0195))))
    for c in (0.0005, up(0.0005), dn(0.0005)):
        cs.append((f"dnet={c!r}", dict(bk=dict(dx=0.0, cpos=c, cneg=0.0, prev_net=0.0))))
    for c in (0.05, up(0.05), dn(0.05)):
        cs.append((f"cpos={c!r}", dict(bk=dict(dx=0.0, cpos=c, cneg=c, prev_net=0.0))))
    for c in (f * 0.2, up(f * 0.2), dn(f * 0.2)):
        cs.append((f"cneg={c!r}", dict(bk=dict(dx=0.0, cpos=0.2, cneg=c, prev_net=0.0))))
    for dv in (-0.02, -0.01, -0.003, -0.001, 0.0, 0.001, 0.003, 0.01):
        cs.append((f"vx={-0.005 + dv}", dict(v={0: -0.005 + dv})))
    angs = (3, 4.5, 6, 9, 11, 22, 24, 27, 30, 45) if variant == "train" else (12, 14, 16, 18, 32, 34, 37, 40, 45, 50, 51, 54, 56)
    for axis, name in enumerate(("roll", "pitch", "yaw")):
        for d in angs:
            for s in (1, -1):
                cs.append((f"{name}={s * d}", dict(quat=_quat(axis, s * d))))
    # trunk heights (settled_z is about 0.06 m, init_z 0.2 m): contacts push a lowered trunk back up within a policy step,
    # so the trunk is thrown up to pass init_z + 0.05, and laid on its back to stay below settled_z - 0.03
    for dz, vz in ((-0.09, 0.0), (-0.05, 0.0), (0.06, 1.0), (0.1, 1.0), (0.15, 1.0), (0.06, 2.0), (0.1, 2.0), (0.15, 2.0)):
        cs.append((f"z+={dz} vz={vz}", dict(dz=dz, v={2: vz})))
    for dz, vz in ((-0.05, -1.0), (0.0, -1.0), (0.0, -0.5)):
        cs.append((f"on its back z+={dz} vz={vz}", dict(dz=dz, v={2: vz}, quat=[0.0, 1.0, 0.0, 0.0])))
    cs += [("nan z", dict(q={2: np.nan})), ("inf qvel7", dict(v={7: np.inf})), ("nan qpos9", dict(q={9: np.nan})),
           ("-inf vx", dict(v={0: -np.inf}))]
    tilt = _quat(0, 30.0 if variant == "train" else 40.0)           # past the roll limit (25 / 35 degrees)
    cs += [("rolled + nan qpos9", dict(quat=tilt, q={9: np.nan})), ("rolled + inf qvel7", dict(quat=tilt, v={7: np.inf}))]
    base, u = np.float32(0.375), np.float32(np.spacing(np.float32(0.375)))
    for k in (0, 2, 5, 8, 12, -2, -5, -8, -12):
        for parity in (0, 1):
            cs.append((f"a=0.375{k:+d}ulp p{parity}", dict(margin=np.float32(base + k * u), parity=parity)))
    for k in range(4):
        cs.append((f"random{k}", dict()))
    return cs


def _build_round(variant, env, ref, qs, vs, cases, case_of, rng):
    """Pre-state, action and counter of every env for one round, and the bookkeeping rule of its case."""
    N = env.N
    q0, v0 = qs.copy(), vs.copy()
    a = rng.uniform(-2, 2, (N, env.ad)).astype(np.float32)
    counter = rng.integers(0, 200, N)
    last = np.tile(ref.home_ctrl32, (N, 1)).astype(np.float64) + rng.uniform(-0.3, 0.3, (N, 8)).astype(np.float32)
    last = last.astype(np.float32).astype(np.float64)
    rules = []
    for i in range(N):
        name, sp = cases[case_of[i]]
        for j, x in sp.get("q", {}).items():
            q0[i, j] = x
        for j, x in sp.get("v", {}).items():
            v0[i, j] = x
        if "quat" in sp:
            q0[i, 3:7] = sp["quat"]
        if "dz" in sp:
            q0[i, 2] = qs[i, 2] + sp["dz"]
        if "margin" in sp:
            counter[i] = 2 * (counter[i] // 2) + sp["parity"]
            if variant == "train":
                a[i] = [sp["margin"], 0.0, sp["margin"], 0.0]
        rules.append(sp.get("bk", dict(dx=float(rng.uniform(-3e-3, 3e-3)), cpos=0.03, cneg=0.01, prev_net=0.0195)))
    return q0, v0, a, counter, last, rules


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("variant", VARIANTS)
def test_post_physics_logic_matches_the_reference(variant, N):
    env = _Env(variant, N)
    qs, vs = env.state()
    ref = _Ref(variant, qs[0, 2])
    if variant == "train":                           # the 40-degree rule is unreachable: ctrlrange bounds every target
        reach = max(DEG * max(abs(lo - h), abs(hi - h)) for (lo, hi), h in zip(ref.o.ctrlrange, ref.home))
        assert reach < 40.0, reach
    cases = _cases(variant)
    K = len(cases)
    idx = _sample(N)
    rng = np.random.default_rng(1000 + N)
    st = _Stats()
    for rnd in range(-(-K // N)):
        case_of = (np.arange(N) + rnd * N) % K
        q0, v0, a, counter, last, rules = _build_round(variant, env, ref, qs, vs, cases, case_of, rng)
        # pass 1: the post-physics x' of this pre-state (the command, hence the physics, depends on the counter's parity)
        env.set_state(q0, v0)
        env.set_bk(dict(counter=counter, prev_x=np.zeros(N), cpos=np.zeros(N), cneg=np.zeros(N), prev_net=np.zeros(N), last_cmd=last))
        env.step(a)
        q1, v1 = env.state()
        bk = _bk_new(N)
        bk["counter"][:] = counter; bk["last_cmd"][:] = last
        for i in range(N):
            x = float(q1[i, 0])
            r = rules[i]
            bk["prev_x"][i] = x - r["dx"]
            bk["cpos"][i], bk["cneg"][i], bk["prev_net"][i] = r["cpos"], r["cneg"], r["prev_net"]
        # pass 2: the same pre-state again, now with the chosen bookkeeping
        env.set_state(q0, v0)
        env.set_bk(bk)
        out = env.step(a)
        q2, v2 = env.state()
        assert _same_bits(q1, q2) and _same_bits(v1, v2), "the replayed step did not repeat the post-physics state"
        last_gpu = last.copy()
        _check_step(variant, ref, out, q2, v2, bk, last_gpu, a, idx, f"{variant} N={N} round {rnd} step 0", st)
        for t in range(1, 3):                        # chained: the oracle carries its own bookkeeping
            a = rng.uniform(-2, 2, (N, env.ad)).astype(np.float32)
            out = env.step(a)
            q, v = env.state()
            _check_step(variant, ref, out, q, v, bk, last_gpu, a, idx, f"{variant} N={N} round {rnd} step {t}", st)
    ang = np.array(st.pop("ang")); z = np.array(st.pop("z")); vx = np.array(st.pop("vx"))
    thr = (5, 10, 25) if variant == "train" else (15, 35, 52.5)
    for t in thr:
        for col in range(3):
            assert (ang[:, col] > math.radians(t)).any() and (ang[:, col] < math.radians(t)).any(), (t, col)
    assert (vx < -0.005).any() and (vx > -0.005).any()
    assert st["reason1"] > 0 and st["reason2"] > 0 and st["reason3"] > 0
    assert st["mj_error_with_orientation"] > 0, "no non-finite state met the orientation rule"
    if variant == "terrain":
        zs = z - ref.o.settled_z; zi = z - ref.o.initial_z_flat
        assert (zs < -0.03).any() and (zs > -0.03).any() and (zi > 0.05).any() and (zi < -0.05).any() and (abs(zi) < 0.05).any()
    else:
        assert st["margin_inside"] > 0 and st["margin_just_outside"] > 0
    print(f"{variant} N={N}: {st.counts()}")


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("variant", VARIANTS)
def test_episode_ends_auto_reset_to_a_fresh_episode(variant, N):
    """The max_steps cap and termination-driven auto-resets, against a twin handle without auto-reset that gives the
    post-physics state of the same pre-state (set_state zeroes both warm starts, so the physics repeats bit for bit)."""
    A = _Env(variant, N, auto_reset=True)            # the trainer's default cap: 250 / 1000
    B = _Env(variant, N)
    qs, vs = A.state()
    reset_obs = A.reset()[0].copy()
    ref = _Ref(variant, qs[0, 2])
    idx = _sample(N)
    rng = np.random.default_rng(77 + N)
    ms = MAX_STEPS[variant]
    # env kinds by index: 0 capped, 1 capped + tilted (termination wins), 2 tilted, 3 backward, 4 non-finite, 5 running
    kind = np.arange(N) % 6 if N > 1 else np.array([1])
    q0, v0 = qs.copy(), vs.copy()
    tilt = _quat(0, 40.0 if variant == "train" else 60.0)
    q0[(kind == 1) | (kind == 2), 3:7] = tilt
    q0[kind == 4, 2] = np.nan
    counter = rng.integers(0, ms - 2, N)            # running envs stay below the cap for two steps
    counter[(kind == 0) | (kind == 1)] = ms - 1
    bk = dict(counter=counter, prev_x=qs[:, 0].astype(np.float64), cpos=np.full(N, 0.01), cneg=np.zeros(N), prev_net=np.zeros(N),
              last_cmd=np.tile(ref.home_ctrl32, (N, 1)).astype(np.float64))
    bk["cpos"][kind == 3] = 0.2; bk["cneg"][kind == 3] = 0.2
    a = rng.uniform(-1, 1, (N, A.ad)).astype(np.float32)
    for E in (A, B):
        E.set_state(q0, v0)
        E.set_bk(bk)
    out = A.step(a)
    outB = B.step(a)
    qB, vB = B.state()
    capped = (bk["counter"] + 1) >= ms
    st = _Stats()
    last_gpu = bk["last_cmd"].copy()
    bk_ref = {k: np.array(v, copy=True) for k, v in bk.items()}
    _check_step(variant, ref, out, qB, vB, bk_ref, last_gpu, a, idx, f"{variant} N={N} episode end", st,
                expect_done=capped, reset_obs=reset_obs)
    done = out["done"].astype(bool)
    assert np.array_equal(done, (out["reason"] > 0) | capped), "done = a termination or the cap"
    assert done[kind <= 1].all() and (out["reason"][kind == 0] == 0).all()
    assert np.array_equal(out["obs"][done], np.broadcast_to(reset_obs, out["obs"][done].shape))
    assert (out["reason"][kind == 1] == REASON["orientation_limit"]).all(), "a termination on the capped step wins"
    assert np.array_equal(out["tobs"][~done], out["obs"][~done])
    qA, vA = A.state()
    assert _same_bits(qA[done], np.broadcast_to(qs[0], qA[done].shape)) and _same_bits(vA[done], np.broadcast_to(vs[0], vA[done].shape))
    assert _same_bits(qA[~done], qB[~done]) and _same_bits(vA[~done], vB[~done])
    assert np.array_equal(outB["obs"][~done], out["obs"][~done])
    # the next step: done envs start a fresh episode (counter 0, prev_x = settled x, zero sums, last_cmd = float32 home ctrl)
    for i in np.flatnonzero(done):
        _bk_set_row(bk_ref, i, dict(counter=0, prev_x=float(qs[0, 0]), cpos=0.0, cneg=0.0, prev_net=0.0,
                                    last_cmd=ref.home_ctrl32.astype(np.float64)))
        last_gpu[i] = ref.home_ctrl32
    a = rng.uniform(-0.5, 0.5, (N, A.ad)).astype(np.float32)
    out = A.step(a)
    q, v = A.state()
    assert not out["done"][done].any()
    _check_step(variant, ref, out, q, v, bk_ref, last_gpu, a, idx, f"{variant} N={N} fresh episode", st)
    assert st["reason0"] > 0
    print(f"{variant} N={N}: {int(done.sum())} episode ends, {st.counts()}")


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("variant", VARIANTS)
def test_masked_reset(variant, N):
    env = _Env(variant, N)
    fresh = _Env(variant, N)
    qs, vs = fresh.state()
    reset_obs = fresh.reset()
    ref = _Ref(variant, qs[0, 2])
    idx = _sample(N)
    rng = np.random.default_rng(5 + N)
    masks = [np.zeros(N, np.uint8), np.ones(N, np.uint8), (rng.random(N) < 0.5).astype(np.uint8)]
    st = _Stats()
    for mi, mask in enumerate(masks):
        env.reset()
        for _ in range(2):                            # move away from the settled state
            env.step(rng.uniform(-1, 1, (N, env.ad)).astype(np.float32))
        bk = dict(counter=rng.integers(0, 200, N), prev_x=rng.uniform(-0.1, 0.1, N), cpos=rng.uniform(0, 0.04, N),
                  cneg=rng.uniform(0, 0.02, N), prev_net=rng.uniform(0, 0.02, N),
                  last_cmd=(np.tile(ref.home_ctrl32, (N, 1)) + rng.uniform(-0.2, 0.2, (N, 8))).astype(np.float32).astype(np.float64))
        env.set_bk(bk)
        q1, v1 = env.state()
        obs = env.reset(mask)
        m = mask.astype(bool)
        sent = env.out["obs"].is_sentinel()
        assert sent[~m].all(), "an unmasked env's obs row was written"
        assert np.array_equal(obs[m], np.broadcast_to(reset_obs[0], obs[m].shape))
        q2, v2 = env.state()
        assert _same_bits(q2[m], qs[m]) and _same_bits(v2[m], vs[m])
        assert _same_bits(q2[~m], q1[~m]) and _same_bits(v2[~m], v1[~m])
        last_gpu = bk["last_cmd"].copy()
        for i in np.flatnonzero(m):
            _bk_set_row(bk, i, dict(counter=0, prev_x=float(qs[0, 0]), cpos=0.0, cneg=0.0, prev_net=0.0,
                                    last_cmd=ref.home_ctrl32.astype(np.float64)))
            last_gpu[i] = ref.home_ctrl32
        a = rng.uniform(-1, 1, (N, env.ad)).astype(np.float32)
        out = env.step(a)
        q, v = env.state()
        _check_step(variant, ref, out, q, v, bk, last_gpu, a, idx, f"{variant} N={N} mask {mi}", st)
    print(f"{variant} N={N}: {st.counts()}")


def _flat_predicted(seed, gid, gen):
    """The generator's flat / rough draw (odg_terrain.cu): word 0 of Philox(seed; gid, gen, 0xFFFFFFFF, "TERR"),
    u01 < 0.5 <=> the word < 2^31."""
    h = _philox_np(seed, gid, gen, 0xFFFFFFFF, 0x54455252)
    return h[0] < np.uint32(0x80000000)


@pytest.mark.parametrize("N", NS)
def test_terrain_fields_follow_the_episode_keying(N):
    from opendog_b200.compat import BatchedTerrainQuadrupedEnv
    seed = 0x1234_5678_9ABC
    rng = np.random.default_rng(9 + N)
    mask = (rng.random(N) < 0.5).astype(np.uint8)
    if N > 1:
        mask[0], mask[-1] = 1, 0
    capped = (rng.random(N) < 0.5)
    if N > 1:
        capped[0], capped[-1] = False, True
    ms = MAX_STEPS["terrain"]

    def run(n, first, sl):
        e = BatchedTerrainQuadrupedEnv(n, seed=seed, first_env_id=first, auto_reset=True)
        gid = np.arange(first, first + n)
        gen = np.zeros(n, np.int64)
        hist = []
        e.reset(); gen += 1
        hist.append(e.hfield_data.cpu().numpy().copy())
        assert np.array_equal((hist[-1] == 0.5).all(1), _flat_predicted(seed, gid, gen - 1))
        for m in (np.zeros(n, np.uint8), mask[sl], np.ones(n, np.uint8)):
            e.reset(torch.from_numpy(m))
            gen += m
            f = e.hfield_data.cpu().numpy().copy()
            mb = m.astype(bool)
            assert np.array_equal(f[~mb], hist[-1][~mb]), "a field outside the mask changed"
            assert np.array_equal((f[mb] == 0.5).all(1), _flat_predicted(seed, gid[mb], gen[mb] - 1))
            both_flat = (f == 0.5).all(1) & (hist[-1] == 0.5).all(1)
            assert ((f != hist[-1]).any(1) | both_flat)[mb].all(), "a regenerated field repeats its predecessor"
            hist.append(f)
        cnt = np.where(capped[sl], ms - 1, 0)
        e.set_bookkeeping(counter=torch.from_numpy(cnt.astype(np.int32)))
        _, _, done, info = e.step(torch.zeros(n, 8))
        done = done.cpu().numpy()
        assert np.array_equal(done, capped[sl]) and (info["termination_reason"].cpu().numpy() == 0).all()
        gen += done
        f = e.hfield_data.cpu().numpy().copy()
        assert np.array_equal(f[~done], hist[-1][~done])
        assert np.array_equal((f[done] == 0.5).all(1), _flat_predicted(seed, gid[done], gen[done] - 1))
        both_flat = (f == 0.5).all(1) & (hist[-1] == 0.5).all(1)
        assert ((f != hist[-1]).any(1) | both_flat)[done].all()
        hist.append(f)
        e.close()
        return hist

    whole = run(N, 0, slice(0, N))
    if N > 1:
        n0 = N // 2
        lo, hi = run(n0, 0, slice(0, n0)), run(N - n0, n0, slice(n0, N))
        for a, b, c in zip(whole, lo, hi):
            assert np.array_equal(a, np.concatenate([b, c])), "two shards do not reproduce the batch's fields"
