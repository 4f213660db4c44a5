"""Host logic: model compiler vs the committed asset, C struct layouts, and the C-ABI library surface."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_committed_asset_has_the_reference_model_constants():
    """The OpenDOG asset against values read off the reference's MJCF (our_robot.xml). Re-deriving the whole asset
    needs that MJCF and its meshes, which are not part of this repository (tools/compile_model.py does it)."""
    from opendog_b200.model.compile import load_compiled
    asset = load_compiled("our_robot")
    assert asset["nq"] == 15 and asset["nv"] == 14 and asset["nu"] == 8 and asset["ngeom"] == 12
    assert abs(asset["base_mass"] + np.sum(asset["mass"]) - 1.95852) < 1e-12       # SURVEY A.1 total mass
    assert asset["act_leg"] == [1, 1, 3, 3, 0, 0, 2, 2]                            # our_robot.xml:99-111
    assert [g["mj_body_id"] for g in asset["geoms"] if g["link"] == 1][1::2] == [4, 7, 10, 13]
    # floor (condim 3, friction 1) wins the max-mixing against the robot geoms (condim 1, friction .6)
    assert all(g["condim"] == 3 and g["friction"] == 1.0 and g["margin"] == 0.001 for g in asset["geoms"])
    assert asset["base_armature"] == [0.02] * 6 and asset["base_frictionloss"] == [0.1] * 6


def test_struct_layouts_match_the_c_headers():
    from oracle import oracle
    oracle.lib()          # asserts sizeof(OdgModel / OdgoData / OdgoWalkEnv) against the compiled C


def test_libodgsim_exports_every_declared_symbol():
    from opendog_b200 import build, lib
    build.build()
    L = C.CDLL(lib.LIB_PATH)
    declared = set()
    for h in sorted(os.listdir(os.path.join(ROOT, "include"))):          # every include/*.h
        header = open(os.path.join(ROOT, "include", h)).read()
        declared |= set(re.findall(r"\b(odg_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    assert declared == set(lib.SYMBOLS), declared ^ set(lib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s


def test_no_cpu_fallback():
    """Without a CUDA device the product path must fail loudly (ODG_ERR_NO_DEVICE), not compute."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from opendog_b200 import lib
    from opendog_b200.model.compile import load_compiled, to_struct
    L = lib.load()
    m = to_struct(load_compiled("our_robot"))
    h = C.c_void_p()
    rc = L.odg_create(C.byref(m), None, 4, 0, 0, C.byref(h))
    assert rc == -3 and b"no CPU fallback" in L.odg_last_error()
    from opendog_b200.env import BatchedWalkEnv
    with pytest.raises(lib.OdgError):
        BatchedWalkEnv(4)


def test_default_config_is_the_references_constants():
    from opendog_b200 import lib
    cfg = lib.OdgEnvConfig()
    lib.load().odg_default_config(C.byref(cfg))
    assert (cfg.frame_skip, cfg.max_episode_steps, cfg.auto_reset, cfg.scale_actions) == (10, 750, 1, 1)
    assert abs(cfg.reset_noise_scale - 0.02) < 1e-9


def test_c_abi_error_behaviour():
    """The boundary never throws or exits: bad arguments come back as negative OdgStatus codes with a message from
    odg_last_error(), and queries on a null handle return 0 (include/odg.h). No device work is issued here."""
    from opendog_b200 import lib
    from opendog_b200.model.compile import load_compiled, to_struct
    L = lib.load()
    m = to_struct(load_compiled("our_robot"))
    h = C.c_void_p()
    INVALID = -1
    assert L.odg_create(None, None, 4, 0, 0, C.byref(h)) == INVALID and b"odg_create" in L.odg_last_error()
    assert L.odg_create(C.byref(m), None, 0, 0, 0, C.byref(h)) == INVALID
    assert L.odg_create(C.byref(m), None, 4, 0, 0, None) == INVALID
    assert L.odg_step(None, None, None, None, None, None, None, None) == INVALID and b"odg_step" in L.odg_last_error()
    assert L.odg_evaluate(None, None, None, None, None, None, None, None) == INVALID
    assert L.odg_step_host(None, None, None, None, None, None, None, None, None, None, None, 0, None) == INVALID and b"odg_step_host" in L.odg_last_error()
    assert L.odg_reset(None, None, None, None) == INVALID and b"odg_reset" in L.odg_last_error()
    assert L.odg_get_state(None, None, None, None) == INVALID
    assert L.odg_set_frame_skip(None, 10) == INVALID
    assert (L.odg_num_envs(None), L.odg_obs_dim(None), L.odg_act_dim(None), L.odg_nq(None), L.odg_nv(None)) == (0,) * 5
    assert L.odg_launch_count(None) == 0
    L.odg_destroy(None)                                   # a no-op, like free(NULL)
    assert L.odg_policy_create(1000, 8, 0, C.byref(h)) < 0      # state_dim above ODG_POLICY_MAX_STATE
    assert L.odg_policy_forward(None, None, 16, None, None, None, None, 0, 0, None, 0, None) < 0
    L.odg_policy_destroy(None)
    # update-phase entry points (include/odg_policy.h): argument checks come before any device work
    assert L.odg_ppo_loss(*([None] * 7), 16, 8, 0.2, 0.5, 0.005, *([None] * 7)) == INVALID and b"odg_ppo_loss" in L.odg_last_error()
    assert L.odg_tanh_bf16(None, None, 64, None) == INVALID and b"odg_tanh_bf16" in L.odg_last_error()
    assert L.odg_tanh_backward_bias(None, None, None, None, None, 4, 512, None) == INVALID
    # the bf16 tensors are moved as 16-byte vectors: a misaligned pointer is refused before any CUDA call (these addresses
    # are never dereferenced)
    A16, A8 = C.c_void_p(0x2000), C.c_void_p(0x1008)
    assert L.odg_tanh_bf16(A8, A16, 64, None) == INVALID and b"16-byte aligned" in L.odg_last_error()
    assert L.odg_tanh_bf16(A16, A8, 64, None) == INVALID and b"16-byte aligned" in L.odg_last_error()
    assert L.odg_tanh_bf16(C.c_void_p(0x2002), C.c_void_p(0x2002), 64, None) == INVALID
    for k in range(3):
        bf = [A8 if i == k else A16 for i in range(3)]
        assert L.odg_tanh_backward_bias(*bf, A16, A16, 4, 512, None) == INVALID
        assert b"odg_tanh_backward_bias" in L.odg_last_error() and b"16-byte aligned" in L.odg_last_error()
    assert L.odg_tanh_backward_bias_scratch_floats(512) >= 512 and L.odg_tanh_backward_bias_scratch_floats(0) == 0
    assert L.odg_ppo_loss_scratch_floats() > 0
    assert L.odg_s2r_step(None, None, None, None, None, None, None, None, None) < 0
    L.odg_s2r_destroy(None)
    assert isinstance(L.odg_version(), bytes) and L.odg_version()
