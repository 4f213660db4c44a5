"""The step kernel's Newton solve (odg_core.cuh: substep) against the fp64 optimum of the same problem, state by state.

The kernel's qacc is meant to minimise the convex Gauss + constraint cost the oracle evaluates in fp64
(`Sim.cost`, odgo_constraint_cost), whose minimiser a* the oracle returns (held to that by test_oracle_physics.py).
The cost's Hessian is at least M, so the cost gap bounds the error in the M-norm:

    1/2 |a - a*|_M^2  <=  gap(a) = cost(a) - cost(a*).

Every state is an oracle state rounded to float32 and stepped once (frame_skip = 1); the kernel's qacc is read from
info["qacc"]. Checks on EVERY state, no outlier quota:
  (a) convergence: solver_iters < solver_iterations;
  (b) optimality: gap <= K * B, and gap >= -(fp64 rounding of the two cost evaluations);
  (c) stopping rule: |a - a_ref|_inf <= tol * (1 + |a_ref|_inf), a_ref from REFERENCE (itself converged before its cap)
      on the same backend;
  (d) (a)-(c) for every line-search setting of LS_GRID.
The only exemptions: a contact-count mismatch that the oracle confirms as a decision within FLIP_M of flipping (counted,
and the count is capped), and the states pinned by index in STOPS_EARLY and NEEDS_ALL_ITERATIONS, which are held to
looser explicit bounds (see there).

B is the float32 floor of the state (see `_oracle_data`): the analytic part is what rounding the forces and the
constraint residuals to float32 costs, the empirical part the largest gap that rounding the STATE by one ulp gives the
oracle's own optimum. The empirical part is what covers Go1: its condim-6 feet have rolling rows with D ~ 1e-2 next to
sliding rows with D ~ 1e2, the cost is that flat along the rolling directions, and a one-ulp change of qpos / qvel moves
the fp64 optimum by a gap of the same size as the kernel's (within 1-7x on the worst states), while the analytic part
misses it by up to 500x. So the kernel and the oracle solve the same problem there; the tail is rounding.
"""
import ctypes as C
import copy
import json
import os
import tempfile

import numpy as np
import pytest

from emu import EmuEnv, OdgEnvConfig, lib as emu_lib
from oracle.oracle import Sim
from opendog_b200.model.compile import load_compiled, to_struct
from test_emu_parity import FLIP_M
from test_gpu_parity import SHAPES, _oracle_rollout_states

EPS = 2.0 ** -24
DEFAULT = dict(solver_iterations=30, solver_tolerance=1e-4)            # odg_default_config's solver settings
REFERENCE = dict(solver_iterations=100, solver_tolerance=1e-6)
LS_GRID = [(n, t) for n in (3, 4, 8) for t in (0.01, 0.1, 0.5)]
MODELS = ("our_robot", "our_robot_condim1", "go1")
SIZES = {"emu": dict(rollout=64, stance=4, condim1=32), "gpu": dict(rollout=2048, go1=1024, stance=64, condim1=512)}

# K: gap / B bound per model and solver setting. "default" covers tol 1e-4 at every LS_GRID setting, where the stopping
# rule, not rounding, sets the gap (an iteration whose full step is short stops before the quadratic phase: OpenDOG
# rollout state 30 stops after 3 iterations 2500x above its converged gap). Measured maxima of gap / B over every state
# except the pinned STOPS_EARLY ones (whose own maximum is given there) and the confirmed contact-count flips:
#   emulator (g++ -ffp-contract=off), its sets: default and every LS_GRID setting OpenDOG 373, condim-1 6.7, Go1 3.7;
#     REFERENCE OpenDOG 5.3, condim-1 6.7, Go1 3.7
#   NVIDIA B200 (1000 W power limit), GPU-sized sets, 2026-10-21: default and every LS_GRID setting OpenDOG 1.24e4
#     (rollout state 1625), condim-1 3.0, Go1 1.42e4 (ls 3 / 0.1; 1.9e3 at the default setting); REFERENCE OpenDOG 5.3,
#     condim-1 3.0, Go1 8.8
# K = 5e4 leaves 3.5x over the largest default-tolerance maximum, 30 leaves 3.4x over the largest reference maximum.
K = {("our_robot", "default"): 5e4, ("our_robot_condim1", "default"): 5e4, ("go1", "default"): 5e4,
     ("our_robot", "reference"): 30.0, ("our_robot_condim1", "reference"): 30.0, ("go1", "reference"): 30.0}

# The known defect of test_short_newton_step_stops_within_the_stopping_rule, pinned by index into the (seeded) state
# sets: at solver_tolerance 1e-4 these states stop beyond the stopping rule's bound of the converged reference, at some
# LS_GRID settings or all of them (790, 1620, 1205 and 1684 at ls_tolerance 0.5 only; 1684 on the B200, where it ends
# at the iteration cap, see NEEDS_ALL_ITERATIONS). Nowhere else may a state do so. They are held to
# STOPS_EARLY_FACTOR times that bound (measured up to 54x: OpenDOG 1059) and to gap / B <= K_STOPS_EARLY (measured up
# to 1.3e7: Go1 316) instead; at the REFERENCE setting they keep the bounds of every other state. The emulator's sets
# have none.
STOPS_EARLY = {("gpu", "our_robot"): (221, 790, 1059, 1620, 1684, 2292), ("gpu", "go1"): (316, 547, 1205)}
STOPS_EARLY_FACTOR = 100.0
K_STOPS_EARLY = 5e7
# States that need all 30 iterations at ls_tolerance 0.5, pinned by index (a random +-1e3 warm start; Go1 1205 is also
# one of STOPS_EARLY). Only (a) is waived for them, and only at ls_tolerance 0.5.
NEEDS_ALL_ITERATIONS = {("emu", "our_robot"): (89,), ("gpu", "our_robot"): (1684,), ("gpu", "go1"): (1205,)}


# ---------------------------------------------------------------------------------------------------------- state sets
def _go1_rollout(n, seed=0):
    """States of an oracle trajectory of Go1 under targets key_ctrl +- 0.3 rad (new targets every 40 substeps, a state
    every 9th substep, back to the keyframe every 1800 substeps so that stand-ups recur)."""
    rng = np.random.default_rng(seed)
    s = Sim("go1")
    s.reset_keyframe()
    lo = np.array([r[0] for r in s.desc["act_ctrlrange"]]); hi = np.array([r[1] for r in s.desc["act_ctrlrange"]])
    mid = np.array(s.desc["key_ctrl"])
    out, k = [], 0
    while len(out) < n:
        if k % 40 == 0:
            s.ctrl[:] = np.clip(mid + rng.uniform(-0.3, 0.3, 12), lo, hi)
        s.step()
        k += 1
        if k % 9 == 0:
            out.append((s.qpos.copy(), s.qvel.copy(), s.qacc_warmstart.copy(), s.ctrl.copy()))
        if k % 1800 == 0:
            s.reset_keyframe()
    return out


def _edge_states(model, base, n_stance, seed):
    """From the first `n_stance` states of `base` with at least two contacts: flight (trunk lifted, no contact: the
    problem is unconstrained and qacc = qacc_smooth), sliding at +-1.5 m/s (cone surface), at rest (sticking), lift-off
    (contacts inside the margin that carry no force), impact (down at up to 2 m/s with a few mm of penetration: stiff
    rows switching on next to the iterate) and joints pushed past their limits (limit rows active)."""
    rng = np.random.default_rng(seed)
    sim = Sim(model)
    njl = sim.desc["njl"]
    lim = np.array(sim.desc["jnt_limited"], bool)[:, :njl].ravel()
    jr = np.array(sim.desc["jnt_range"])[:, :njl]
    rng_lo, rng_hi = jr[..., 0].ravel(), jr[..., 1].ravel()
    out = []
    for q, v, w, c in base:
        if len([s for s in out if s[0] == "flight"]) == n_stance:
            break
        _set(sim, q, v, w, c)
        sim.forward()
        if sim.ncon < 2:
            continue
        q1 = q.copy(); q1[2] += 0.5
        out.append(("flight", (q1, v, w, c)))
        for sgn in (1.0, -1.0):
            v1 = v.copy(); v1[len(out) % 2] = 1.5 * sgn
            out.append(("sliding", (q, v1, w, c)))
        out.append(("rest", (q, np.zeros_like(v), w, c)))
        v1 = v.copy(); v1[2] = 0.4
        out.append(("lift-off", (q, v1, w, c)))
        q1 = q.copy(); q1[2] -= rng.uniform(1e-3, 4e-3); v1 = v.copy(); v1[2] = -rng.uniform(0.5, 2.0)
        out.append(("impact", (q1, v1, w, c)))
        # (only bounds within 0.5 rad of the pose: a Go1 thigh at its 4.5 rad bound folds the leg deep into the floor)
        q1 = q.copy()
        for j in np.flatnonzero(lim):
            near_lo = q[7 + j] - rng_lo[j] < rng_hi[j] - q[7 + j]
            bound = rng_lo[j] if near_lo else rng_hi[j]
            if rng.uniform() < 0.5 and abs(bound - q[7 + j]) < 0.5:
                q1[7 + j] = bound - rng.uniform(0, 0.03) if near_lo else bound + rng.uniform(0, 0.03)
        if np.array_equal(q1, q):                    # none drawn: the joint nearest to a bound goes 0.01 rad past it
            d_lo, d_hi = q[7:][lim] - rng_lo[lim], rng_hi[lim] - q[7:][lim]
            k = np.argmin(np.minimum(d_lo, d_hi)); j = np.flatnonzero(lim)[k]
            q1[7 + j] = rng_lo[j] - 0.01 if d_lo[k] < d_hi[k] else rng_hi[j] + 0.01
        out.append(("limits", (q1, v, w, c)))
    assert len([s for s in out if s[0] == "flight"]) == n_stance
    return out


def _set(sim, q, v, w, c):
    sim.reset_keyframe()
    sim.qpos[:] = q; sim.qvel[:] = v; sim.qacc_warmstart[:] = w; sim.ctrl[:] = c


def _condim1_desc():
    """The model variant of test_frictionless_rows_go_through_the_cone_block: every contact condim 1."""
    desc = copy.deepcopy(load_compiled("our_robot"))
    for g in desc["geoms"]:
        g["condim"] = 1
    return desc


_PROBLEMS = {}


def _problem(model, backend):
    """States (float32), labels and the oracle's data for one model and backend size. Warm starts rotate over the
    oracle trajectory's own, zeros, qacc_smooth, the oracle optimum and random +-1e3."""
    key = (model, backend)
    if key in _PROBLEMS:
        return _PROBLEMS[key]
    sz = SIZES[backend]
    desc = _condim1_desc() if model == "our_robot_condim1" else load_compiled(model)
    if model == "go1":
        base = _go1_rollout(sz.get("go1", sz["rollout"]))
    else:
        base = _oracle_rollout_states(sz["condim1"] if model == "our_robot_condim1" else sz["rollout"], seed=1)
    sim_model = desc if model == "our_robot_condim1" else model
    labeled = [("rollout", s) for s in base]
    if model != "our_robot_condim1":
        labeled += _edge_states(sim_model, base, sz["stance"], seed=3)
    labels = np.array([l for l, _ in labeled])
    f32 = lambda i: np.stack([s[i] for _, s in labeled]).astype(np.float32)
    q, v, w, c = f32(0), f32(1), f32(2), f32(3)
    d = _oracle_data(sim_model, q, v, w, c)
    rng = np.random.default_rng(7)
    kind = np.arange(len(q)) % 5
    w = w.copy()
    w[kind == 1] = 0
    w[kind == 2] = d["qacc_smooth"][kind == 2]
    w[kind == 3] = d["astar"][kind == 3]
    w[kind == 4] = rng.uniform(-1e3, 1e3, w[kind == 4].shape)
    p = dict(model=model, backend=backend, desc=desc, sim_model=sim_model, q=q, v=v, w=w.astype(np.float32), c=c, labels=labels, **d)
    _PROBLEMS[key] = p
    return p


def _oracle_data(sim_model, q, v, w, c, trials=4):
    """a*, its cost, ncon and decision gaps, and the float32 floor B = B_an + B_ulp of every state. With eps = 2^-24:
    B_an = 1/2 g' M^-1 g + 1/2 sum_r D_r (eps s_r)^2, g = eps (|M||a*| + |qfrc_bias| + |qfrc_actuator|),
    s_r = |J_r||a*| + |aref_r|; B_ulp = the largest cost gap of the oracle's optimum for the state with every qpos / qvel
    component moved one float32 ulp up or down (`trials` seeded sign patterns that keep the contact count)."""
    sim, sp = Sim(sim_model), Sim(sim_model)
    rng = np.random.default_rng(0)
    n = len(q)
    out = dict(astar=np.zeros((n, sim.nv)), cstar=np.zeros(n), scale=np.zeros(n), ncon=np.zeros(n, int),
               flip=np.zeros(n, bool), nlim=np.zeros(n, int), B=np.zeros(n), B_an=np.zeros(n), qacc_smooth=np.zeros((n, sim.nv)))
    up = lambda x: np.nextafter(x, np.float32(np.inf)); dn = lambda x: np.nextafter(x, np.float32(-np.inf))
    for i in range(n):
        _set(sim, q[i], v[i], w[i], c[i])
        sim.forward()
        a = sim.qacc.copy(); c0 = sim.cost(a); M = sim.M
        g = EPS * (np.abs(M) @ np.abs(a) + np.abs(sim.qfrc_bias) + np.abs(sim.qfrc_actuator))
        s = np.abs(sim.efc_J) @ np.abs(a) + np.abs(sim.efc("aref"))
        b_an = 0.5 * g @ np.linalg.solve(M, g) + 0.5 * np.sum(sim.efc("D") * (EPS * s) ** 2)
        b_ulp = 0.0
        for t in range(trials):
            qp = np.where(rng.uniform(size=q.shape[1]) < 0.5, up(q[i]), dn(q[i]))
            vp = np.where(rng.uniform(size=v.shape[1]) < 0.5, up(v[i]), dn(v[i]))
            _set(sp, qp, vp, w[i], c[i])
            sp.forward()
            if sp.ncon == sim.ncon:
                b_ulp = max(b_ulp, sim.cost(sp.qacc.copy()) - c0)
        out["astar"][i] = a; out["cstar"][i] = c0; out["ncon"][i] = sim.ncon
        out["nlim"][i] = int((sim.efc("type") == 1).sum())            # active joint-limit rows (ODGO_ROW_LIMIT)
        out["scale"][i] = c0 + np.abs(a) @ np.abs(M) @ np.abs(a)
        out["flip"][i] = min(sim.decision_gaps[0], sim.decision_gaps[1]) < FLIP_M
        out["B_an"][i] = b_an; out["B"][i] = b_an + b_ulp
        out["qacc_smooth"][i] = sim.qacc_smooth
    return out


# ------------------------------------------------------------------------------------------------------------ backends
def _run(p, backend, shape="auto", **cfg):
    """One substep of every state: (qacc, solver_iters, ncon)."""
    common = dict(frame_skip=1, scale_actions=0, auto_reset=0, **cfg)
    if backend == "emu":
        env = EmuEnv(len(p["q"]), model=p["desc"], **common)
        env.set_state(p["q"], p["v"], p["w"])
        _, _, _, _, info = env.step(p["c"])
        return info["qacc"].astype(np.float64), info["solver_iters"], info["ncon"]
    import torch
    from opendog_b200.env import BatchedWalkEnv
    if p["model"] == "our_robot_condim1":
        # BatchedWalkEnv takes a builtin name or a .json path; the file is read by the constructor and removed after it
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "our_robot_condim1.json")
            with open(path, "w") as fh:
                json.dump(p["desc"], fh)
            env = BatchedWalkEnv(len(p["q"]), model=path, info_keys=("qacc", "ncon", "solver_iters"), **SHAPES[shape], **common)
    else:
        env = BatchedWalkEnv(len(p["q"]), model=p["model"], info_keys=("qacc", "ncon", "solver_iters"), **SHAPES[shape],
                             **common)
    env.set_state(p["q"], p["v"], p["w"])
    _, _, _, info = env.step(torch.from_numpy(p["c"]).cuda())
    return (info["qacc"].cpu().numpy().astype(np.float64), info["solver_iters"].cpu().numpy(),
            info["ncon"].cpu().numpy())


def _gaps(p, qacc):
    sim = Sim(p["sim_model"])
    gap = np.zeros(len(qacc))
    for i in range(len(qacc)):
        _set(sim, p["q"][i], p["v"][i], p["w"][i], p["c"][i])
        sim.forward()
        gap[i] = sim.cost(qacc[i]) - p["cstar"][i]
    return gap


def _check(p, run, cfg, kclass, ref=None):
    """(a), (b) and, given the reference run, (c) on every state; returns gap / B for the report. The only states held
    to other bounds are the ones pinned by index in STOPS_EARLY (for (b) and (c)) and NEEDS_ALL_ITERATIONS (for (a))."""
    qacc, iters, ncon = run
    mism = ncon != p["ncon"]
    assert not (mism & ~p["flip"]).any(), f"contact count differs without a decision flip: {np.flatnonzero(mism & ~p['flip'])}"
    assert mism.sum() <= 2 + len(qacc) // 1000, f"{mism.sum()} contact-count flips"
    ok = ~mism
    key = (p["backend"], p["model"])
    pinned_cap = np.array(NEEDS_ALL_ITERATIONS.get(key, ()) if cfg.get("ls_tolerance") == 0.5 else (), int)
    capped = np.flatnonzero(ok & (iters >= cfg["solver_iterations"]))
    extra = np.setdiff1d(capped, pinned_cap)
    assert extra.size == 0, f"{cfg}: states at the iteration cap: {extra} ({p['labels'][extra]})"
    gap = _gaps(p, qacc)
    ratio = gap / p["B"]
    low = np.flatnonzero(ok & (gap < -2.0 ** -40 * p["scale"]))
    assert low.size == 0, f"{cfg}: cost below the fp64 optimum at {low}: {gap[low]}"
    pinned_far = np.array(STOPS_EARLY.get(key, ()) if ref is not None else (), int)
    loose = np.zeros(len(qacc), bool); loose[pinned_far] = True
    k = K[(p["model"], kclass)]
    bad = np.flatnonzero(ok & (ratio > np.where(loose, K_STOPS_EARLY, k)))
    assert bad.size == 0, f"{cfg}: gap / B above its bound at {bad} ({p['labels'][bad]}): {ratio[bad]}"
    if ref is not None:
        a_ref = ref[0]
        lim = cfg["solver_tolerance"] * (1 + np.abs(a_ref).max(1)) * np.where(loose, STOPS_EARLY_FACTOR, 1.0)
        far = np.flatnonzero(ok & (np.abs(qacc - a_ref).max(1) > lim))
        assert far.size == 0, f"{cfg}: qacc beyond the stopping rule's bound of the reference at {far} ({p['labels'][far]})"
    return ratio[ok]


BACKENDS = [pytest.param("emu", id="emu"), pytest.param("gpu", id="gpu", marks=pytest.mark.gpu)]
_REF = {}


def _reference(p, backend, shape="auto"):
    key = (p["model"], backend, shape)
    if key not in _REF:
        run = _run(p, backend, shape, **REFERENCE)
        _check(p, run, REFERENCE, "reference")
        _REF[key] = run
    return _REF[key]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("backend", BACKENDS)
def test_newton_solve_reaches_the_fp64_optimum(backend, model):
    """The default solver settings and the reference setting (100 iterations, tol 1e-6) on every state set."""
    p = _problem(model, backend)
    ref = _reference(p, backend)
    _check(p, _run(p, backend, **DEFAULT), DEFAULT, "default", ref)
    assert (p["ncon"][p["labels"] == "flight"] == 0).all()
    for lab in ("sliding", "rest", "lift-off", "impact", "limits") if model != "our_robot_condim1" else ():
        assert (p["labels"] == lab).any()
    if model != "our_robot_condim1":
        assert (p["nlim"][p["labels"] == "limits"] > 0).all(), "a 'limits' state without an active limit row"


@pytest.mark.parametrize("ls_iterations,ls_tolerance", LS_GRID, ids=[f"ls{n}-{t}" for n, t in LS_GRID])
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("backend,shape", [pytest.param("emu", "auto", id="emu"),
                                           pytest.param("gpu", "auto", id="gpu-auto", marks=pytest.mark.gpu),
                                           pytest.param("gpu", "large-batch", id="gpu-large-batch", marks=pytest.mark.gpu)])
def test_line_search_settings_reach_the_same_solution(backend, shape, model, ls_iterations, ls_tolerance):
    """ls_iterations x ls_tolerance change the path of the iteration, not where it stops: (a)-(c) for each setting,
    on the GPU under the two launch shapes the others are held bit-identical to."""
    p = _problem(model, backend)
    cfg = dict(DEFAULT, ls_iterations=ls_iterations, ls_tolerance=ls_tolerance)
    _check(p, _run(p, backend, shape, **cfg), cfg, "default", _reference(p, backend, shape))


@pytest.mark.xfail(strict=True, reason="the step-size exit trusts a short full Newton step taken with the iterate's active "
                                      "set; these states stop 7-30x the stopping rule's bound away from the optimum")
def test_short_newton_step_stops_within_the_stopping_rule():
    """Two states, zero warm start, where the default exit fires on a full step of 6e-5 / 8e-5 of the iterate although
    the iterate is still 1.75 (Go1, |a*| 585) and 0.050 (OpenDOG, |a*| 65) away from the fp64 optimum, beyond
    tol * (1 + |a*|) = 0.059 and 0.0066: the Hessian at the iterate includes rows the optimum does not, so the short step
    underestimates the distance. Making the exit safe changes the default path's results, which is left to a
    solver change of its own."""
    for model, states in (("go1", _go1_rollout(317)[316:]), ("our_robot", _oracle_rollout_states(222, seed=1)[221:])):
        q, v, w, c = [np.stack([s[i] for s in states]).astype(np.float32) for i in range(4)]
        w[:] = 0
        env = EmuEnv(1, model=model, frame_skip=1, scale_actions=0, auto_reset=0, **DEFAULT)
        env.set_state(q, v, w)
        a = env.step(c)[4]["qacc"][0].astype(np.float64)
        astar = _oracle_data(model, q, v, w, c, trials=0)["astar"][0]
        assert np.abs(a - astar).max() <= DEFAULT["solver_tolerance"] * (1 + np.abs(astar).max()), model


def test_fewer_than_three_line_search_passes_are_rejected_by_the_config_check():
    """One pass evaluates phi' only at {0.25, 0.5, 1, 2}: a zero below 0.25 is then approached by the chord across the
    kink on every iteration and the solve ends at the cap unconverged; with two, states of both models still stall at
    the cap (on the B200 up to 1e9x above their float32 floor). odg::prepare refuses both (the emulator runs the same
    check and returns null)."""
    m = to_struct(load_compiled("our_robot"))
    for n, accepted in ((0, False), (1, False), (2, False), (3, True), (4, True)):
        cfg = OdgEnvConfig()
        emu_lib().emu_default_config(C.byref(cfg))
        cfg.ls_iterations = n
        h = emu_lib().emu_create(C.byref(m), C.byref(cfg), 1, 0)
        assert bool(h) == accepted, n
        if h:
            emu_lib().emu_destroy(C.c_void_p(h))


@pytest.mark.gpu
def test_fewer_than_three_line_search_passes_are_rejected_by_odg_create():
    from opendog_b200 import lib as L
    lib = L.load()
    m = to_struct(load_compiled("our_robot"))
    for n, status in ((1, -1), (2, -1), (3, 0)):
        cfg = L.OdgEnvConfig()
        lib.odg_default_config(C.byref(cfg))
        cfg.ls_iterations = n
        h = C.c_void_p()
        assert lib.odg_create(C.byref(m), C.byref(cfg), 4, 0, C.c_uint64(0), C.byref(h)) == status, n
        if h:
            lib.odg_destroy(h)


def _report(backend):
    """Print the gap / B distributions per model and setting: with tests/ and tests/emu on sys.path,
    `import test_solver_optimality as t; t._report("emu" or "gpu")`."""
    for model in MODELS:
        p = _problem(model, backend)
        for shape in (("auto", "large-batch") if backend == "gpu" else ("auto",)):
            for name, cfg in [("reference", REFERENCE), ("default", DEFAULT)] + [
                    (f"ls {n} / {t}", dict(DEFAULT, ls_iterations=n, ls_tolerance=t)) for n, t in LS_GRID]:
                qacc, iters, ncon = _run(p, backend, shape, **cfg)
                gap = _gaps(p, qacc)
                ok = ncon == p["ncon"]
                pinned = np.zeros(len(ok), bool)
                if cfg is not REFERENCE:
                    pinned[list(STOPS_EARLY.get((backend, model), ()))] = True
                r, a = (gap / p["B"])[ok & ~pinned], (gap / p["B_an"])[ok & ~pinned]
                rp = (gap / p["B"])[ok & pinned]
                print(f"{model:18s} {shape:11s} {name:14s} N={ok.sum():5d} iters max {iters[ok].max():3d}  gap/B median "
                      f"{np.median(r):.2f} p99 {np.percentile(r, 99):.1f} max {r.max():.3g}   gap/B_an median {np.median(a):.1f} "
                      f"p99 {np.percentile(a, 99):.0f} max {a.max():.3g}   pinned max {rp.max() if rp.size else 0:.3g}", flush=True)
