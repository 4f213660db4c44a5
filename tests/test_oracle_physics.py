"""The oracle (oracle/odg_oracle.c) against independent checks: a generic numpy rigid-body model,
finite differences, analytic cases, KKT/optimality of the constraint solve, RNG known answers.
The reference has no tests for this path (SURVEY §4), so these are the pins we can make ourselves."""
import numpy as np

from oracle.oracle import Sim, WalkEnv, philox, scale_action


def _generic_model(name="our_robot"):
    """The committed asset's body tree as a generic model for opendog_b200.model.rbd_numpy: world, the trunk on a free
    joint, then every leg as a serial chain of hinge links (welded paws already fused into the last link)."""
    from opendog_b200.model.compile import load_compiled
    from opendog_b200.model.mjcf import Body, Joint, MjcfModel
    d = load_compiled(name)
    a = lambda x: np.array(x, dtype=float)
    unit = a([1, 0, 0, 0])
    bodies = [Body("world", -1, np.zeros(3), unit),
              Body("trunk", 0, np.zeros(3), unit, d["base_mass"], a(d["base_ipos"]), a(d["base_inertia"]).reshape(3, 3), [0])]
    joints = [Joint("root", 1, "free", np.zeros(3), np.zeros(3), False, np.zeros(2), d["base_armature"][0],
                    d["base_damping"][0], d["base_frictionloss"][0], 0.0, 0, 0)]
    for leg in range(d["nleg"]):
        parent = 1
        for k in range(d["njl"]):
            h = len(joints) - 1                                   # hinges before this one
            bodies.append(Body(f"leg{leg}_link{k}", parent, a(d["body_pos"][leg][k]), a(d["body_quat"][leg][k]),
                               d["mass"][leg][k], a(d["ipos"][leg][k]), a(d["inertia"][leg][k]).reshape(3, 3), [len(joints)]))
            joints.append(Joint(f"leg{leg}_joint{k}", len(bodies) - 1, "hinge", a(d["jnt_pos"][leg][k]),
                                a(d["jnt_axis"][leg][k]), bool(d["jnt_limited"][leg][k]), a(d["jnt_range"][leg][k]),
                                d["armature"][leg][k], d["damping"][leg][k], d["frictionloss"][leg][k], 0.0, 7 + h, 6 + h))
            parent = len(bodies) - 1
    return MjcfModel(bodies, joints, [], [], {}, {"gravity": a(d["gravity"])}, d["nq"], d["nv"], d["source"])


def _random_state(sim, rng, spread=0.3):
    sim.reset_keyframe()
    sim.qpos[:] = np.array(sim.desc["key_qpos"]) + rng.uniform(-spread, spread, sim.nq)
    sim.qvel[:] = rng.uniform(-1, 1, sim.nv)


def test_philox_known_answer():
    # Random123 known-answer vectors for philox4x32-10
    assert philox(0, 0, 0, 0, 0) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert philox(0xffffffffffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff) == \
        [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert philox(0x299f31d0a4093822, 0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_mass_matrix_and_kinematics_match_generic_numpy_model():
    from opendog_b200.model import rbd_numpy as rbd
    m = _generic_model()
    sim = Sim()
    rng = np.random.default_rng(0)
    for _ in range(5):
        _random_state(sim, rng)
        sim.kinematics(); sim.mass_matrix()
        q = sim.qpos.copy()
        M = rbd.mass_matrix(m, q)
        assert np.abs(M - sim.M).max() < 1e-13
        assert np.all(np.linalg.eigvalsh(sim.M) > 0) and np.allclose(sim.M, sim.M.T)
        kin = rbd.kinematics(m, q)
        assert np.abs(kin["xpos"][1:10] - sim.xpos[:9]).max() < 1e-14           # trunk, then 4 legs x 2 links


def test_bias_force_matches_finite_difference_newton_euler():
    from opendog_b200.model import rbd_numpy as rbd
    m = _generic_model()
    sim = Sim()
    rng = np.random.default_rng(1)
    for _ in range(3):
        _random_state(sim, rng)
        sim.kinematics(); sim.bias()
        c = rbd.bias_force(m, sim.qpos.copy(), sim.qvel.copy())
        assert np.abs(c - sim.qfrc_bias).max() < 1e-6


def test_free_fall_with_trunk_friction_loss():
    """Airborne, the only constraint rows are the 14 friction-loss rows; the trunk's vertical one saturates
    at 0.1 N, so a_z = -(m g - 0.1) / (m + armature)  (our_robot.xml:10: armature .02, frictionloss .1)."""
    sim = Sim()
    sim.reset_keyframe()
    for _ in range(30):
        sim.step()
    assert sim.ncon == 0 and sim.nefc >= 14
    v0 = sim.qvel[2]
    sim.step()
    a = (sim.qvel[2] - v0) / 0.002
    m = 1.95852
    assert abs(a - (-(m * 9.81 - 0.1) / (m + 0.02))) < 2e-3
    assert abs(np.linalg.norm(sim.qpos[3:7]) - 1) < 1e-14


def test_settles_on_the_floor_carrying_its_weight():
    sim = Sim()
    sim.reset_keyframe()
    for _ in range(1500):
        sim.step()
    fn = sum(c["force"][0] for c in sim.contacts())
    assert abs(fn - 1.95852 * 9.81) < 0.02 * 1.95852 * 9.81
    assert 0.04 < sim.qpos[2] < 0.11                      # reward_calc:86 z_range
    assert np.abs(sim.qvel).max() < 1e-3
    for c in sim.contacts():
        assert c["force"][0] >= 0 and c["dist"] < 0.001
        # friction cone: |f_t| <= mu * f_n with mu = 1 (floor default friction wins the max)
        assert np.hypot(c["force"][1], c["force"][2]) <= c["force"][0] * 1.0 + 1e-9


def test_constraint_solution_is_the_minimiser():
    sim = Sim()
    rng = np.random.default_rng(3)
    sim.reset_keyframe()
    checked = 0
    for k in range(400):
        if k % 20 == 0:
            sim.ctrl[:] = np.array([2.36, -1.8] * 4) + rng.uniform(0, 1, 8) * np.array([.44, .6] * 4)
        sim.step()
        if k > 80 and k % 16 == 0:
            q, v, w, c = sim.qpos.copy(), sim.qvel.copy(), sim.qacc_warmstart.copy(), sim.ctrl.copy()
            sim.forward()
            a = sim.qacc.copy()
            f0 = sim.cost(a)
            # M (a - a_smooth) = J^T f  (stationarity of the primal problem)
            lhs = sim.M @ (a - sim.qacc_smooth)
            assert np.abs(lhs - sim.qfrc_constraint).max() < 1e-7 * max(1.0, np.abs(lhs).max())
            for _ in range(8):
                d = rng.normal(size=sim.nv) * 10 ** rng.uniform(-6, -1)
                assert sim.cost(a + d) >= f0 - 1e-9 * max(1.0, abs(f0))
            checked += 1
            sim.qpos[:] = q; sim.qvel[:] = v; sim.qacc_warmstart[:] = w; sim.ctrl[:] = c
    assert checked > 10


def test_pd_actuator_and_limits():
    """home keyframe: thigh starts 3.8 mrad below its lower limit 2.36 (our_robot.xml:14,115) -> limit rows
    active; ctrl is clamped to ctrlrange; force clamped to +-0.83."""
    sim = Sim()
    sim.reset_keyframe()
    sim.ctrl[:] = 10.0
    sim.forward()
    assert np.allclose(np.abs(np.array(sim.d.actuator_force[:8])), 0.83)
    types = np.array(sim.d.efc_type[:sim.nefc])
    assert (types == 0).sum() == 14 and (types == 1).sum() == 4


def test_scale_action_is_numpy_float32():
    rng = np.random.default_rng(0)
    lo = np.array([2.36, -1.8] * 4, dtype=np.float32); hi = np.array([2.8, -1.20] * 4, dtype=np.float32)
    for _ in range(50):
        a = rng.uniform(-1, 1, 8).astype(np.float32)
        ref = lo + (a + 1.0) * (hi - lo) / 2.0               # ScaleActionEnvironment.py:22
        assert ref.dtype == np.float32
        assert np.array_equal(scale_action(a), ref)


def test_walk_env_episode_semantics():
    e = WalkEnv(seed=5, env_id=3)
    e.e.max_steps = 12
    obs = e.reset()
    assert obs.shape == (33,) and not obs[:6].any() and not obs[17:].any()
    assert 1.0 <= obs[6] <= 2.0 and obs[7] == 0 and obs[8] == 0    # 2 * desired velocity, x in [0.5, 1]
    rng = np.random.default_rng(0)
    for t in range(12):
        a = rng.uniform(-1, 1, 8).astype(np.float32)
        obs, r, done, trunc, tobs, info = e.step_autoreset(a)
        assert r >= 0.0                                           # WalkEnvironment.py:84 clip at zero
        assert done == (t == 11)
    assert trunc and e.e.step == 0 and e.e.episode == 2
    assert not np.array_equal(tobs, obs)
