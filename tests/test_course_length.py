"""CPU: courses of 3 to 32 stones (`AllstepsCfg.num_steps`, CFG:90) -- the parameter's way into the C ABI, the Philox
draw mapping of the thread-per-env stone generator for every course length, and the oracle port at other lengths
(against the live reference where its checkout is mounted)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest
import torch

from allsteps_isaaclab_b200 import _cabi, build
from allsteps_isaaclab_b200.config import AllstepsCfg
from allsteps_isaaclab_b200.params import make_params
from oracle import philox, ref_loader

LENGTHS = (3, 4, 7, 12, 31, 32)


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _cabi.load()


@pytest.mark.parametrize("bad", [0, 1, 2, 33, 64, -1, 12.0, True, "12"])
def test_make_params_refuses_course_lengths_outside_3_to_32(bad):
    with pytest.raises(ValueError, match="num_steps"):
        make_params(AllstepsCfg(num_steps=bad))


def test_make_params_sets_num_steps_and_the_struct_keeps_its_layout():
    for S in (3, 20, 32, np.int64(12)):
        assert make_params(AllstepsCfg(num_steps=S)).num_steps == int(S)
    assert AllstepsCfg().num_steps == _cabi.NUM_STONES == 20
    # the field sits in what was the padding between grid_bins and seed: every other offset and the size stay
    assert _cabi.AsParams.grid_bins.offset == 744
    assert _cabi.AsParams.num_steps.offset == 748
    assert _cabi.AsParams.seed.offset == 752
    assert C.sizeof(_cabi.AsParams) == 760


def test_library_validates_the_course_length(lib):
    assert lib.as_sizeof(0) == 760
    p = make_params(AllstepsCfg())
    n = 1 << 20
    # num_steps = 0 is the default length: what a caller that zero-initialises the struct gets
    p.num_steps = 0
    assert lib.as_workspace_bytes_for(C.byref(p), n) == lib.as_workspace_bytes(n)
    p.num_steps = 20
    assert lib.as_workspace_bytes_for(C.byref(p), n) == lib.as_workspace_bytes(n)
    # only the stone rows grow: S x 16 bytes per env
    p.num_steps = 32
    assert lib.as_workspace_bytes_for(C.byref(p), n) - lib.as_workspace_bytes(n) == n * 12 * 16
    p.num_steps = 3
    assert lib.as_workspace_bytes_for(C.byref(p), n) == lib.as_workspace_bytes(n) - n * 17 * 16
    h = C.c_void_p()
    for bad in (1, 2, 33, 0xFFFFFFFF):
        p.num_steps = bad
        assert lib.as_workspace_bytes_for(C.byref(p), n) == 0
        assert lib.as_create(C.byref(p), 64, 0, 0, None, 0, None, C.byref(h)) == -1
        assert b"num_steps" in lib.as_last_error()
    # the workspace is checked against the handle's course length
    p.num_steps = 32
    small = lib.as_workspace_bytes(64)
    raw = np.zeros(small + 256, dtype=np.uint8)
    addr = (raw.ctypes.data + 255) // 256 * 256
    assert lib.as_create(C.byref(p), 64, 0, 0, addr, small, None, C.byref(h)) == -1
    assert b"workspace too small" in lib.as_last_error()


def _philox_block(seed: int, step: int, stream: int, env_id: int, block: int) -> np.ndarray:
    ctr = np.array([env_id, block, step & 0xFFFFFFFF, (stream & 0xFF) | (((step >> 32) & 0xFFFFFF) << 8)],
                   dtype=np.uint32)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    return philox.philox4x32_10(ctr, key)


def kernel_thread_draws(seed: int, step: int, env_id: int, S: int) -> np.ndarray:
    """(3,S): the uniforms k_reset_rows' thread-per-env generator hands to stone s, modelled step by step on its draw
    lambda -- the three cached blocks are fetched together at the first stone and whenever draw k*S+s of any k starts a
    new block, and draw k*S+s is lane (k*S+s) & 3 of the cached block k."""
    out = np.zeros((3, S), dtype=np.float32)
    blk = [None, None, None]
    for s in range(S):
        for k in range(3):
            if k == 0 and (s == 0 or s % 4 == 0 or (S + s) % 4 == 0 or (2 * S + s) % 4 == 0):
                blk = [_philox_block(seed, step, philox.STREAM_STONES, env_id, (q * S + s) >> 2) for q in range(3)]
            d = k * S + s
            assert blk[k] is not None and (d >> 2) == ((k * S + s) >> 2)
            out[k, s] = philox.u32_to_unit_float(blk[k][d & 3:(d & 3) + 1])[0]
    return out


@pytest.mark.parametrize("S", range(3, 33))
def test_thread_generator_draw_mapping_is_the_stone_tables(S):
    seed, step = 0x1234_5678_9ABC, (7 << 32) + 11
    ids = np.array([0, 5, 4_000_001], dtype=np.int64)
    tables = philox.stone_tables(seed, step, ids, S)
    assert tables.shape == (5, 3, S)
    for i, gid in enumerate(ids):
        np.testing.assert_array_equal(kernel_thread_draws(seed, step, int(gid), S), tables[:3, i])


def _replay_to_the_end(S: int, num_envs: int = 256, steps: int = 14, seed: int = 77):
    from oracle import allsteps_oracle as ao
    from scenario import Scenario, install_mdp_state

    sc = Scenario(num_envs, seed=seed, cfg=AllstepsCfg(num_steps=S))
    st0 = sc.initial_mdp_state()
    st0["curr_target_index"] = torch.randint(max(S - 3, 1), S, (num_envs,), generator=sc.gen)
    orc = ao.AllstepsOracle(sc.cfg, num_envs, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    install_mdp_state(orc, st0, num_steps=S)
    return sc, orc


@pytest.mark.parametrize("S", LENGTHS)
def test_oracle_replays_envs_onto_the_last_stone(S):
    sc, orc = _replay_to_the_end(S)
    assert tuple(orc.steps_pos.shape) == (sc.N, S, 3) and tuple(orc.steps_dphi.shape) == (sc.N, S)
    # stones 0..2 are the fixed start stones of ENV:144-150: a straight line from the origin
    sep = sc.cfg.init_step_separation
    np.testing.assert_allclose((orc.steps_pos[:, :3] - sc.env_origins[:, None]).numpy(),
                               np.broadcast_to(np.array([[0, 0, 0], [sep, 0, 0], [2 * sep, 0, 0]], np.float32),
                                               (sc.N, 3, 3)), atol=1e-5)
    arrived = 0
    for step in range(14):
        before = orc.curr_target_index.clone()
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(step))
        idx = orc.pass1["curr_target_index"]
        assert int(idx.max()) <= S - 1 and int(idx.min()) >= 0
        arrived += int(((idx == S - 1) & (before == S - 2)).sum())
        assert torch.equal(orc.prev_target_index, torch.clamp(orc.curr_target_index - 1, 0, S - 1))
        assert torch.equal(orc.next_target_index, torch.clamp(orc.curr_target_index + 1, 0, S - 1))
    assert arrived > 0, "no env stepped from S-2 onto the last stone"


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference checkout not mounted")
@pytest.mark.parametrize("S", [12, 32])
def test_port_is_bit_identical_to_live_reference_at_other_course_lengths(S):
    from allsteps_isaaclab_b200.config import BODY_NAMES, JOINT_NAMES
    from oracle import allsteps_oracle as ao
    from oracle import ref_fake_env as rf
    from scenario import Scenario, install_mdp_state

    num_envs = 128
    sc = Scenario(num_envs, seed=5 + S, full_bodies=True, cfg=AllstepsCfg(num_steps=S))
    su = sc.stone_uniforms(0)
    st0 = sc.initial_mdp_state()
    st0["curr_target_index"] = torch.randint(max(S - 4, 1), S, (num_envs,), generator=sc.gen)
    orc = ao.AllstepsOracle(sc.cfg, num_envs, sc.env_origins, sc.joint_limits, sc.body_indices, su)
    phys = sc.physics(orc.steps_pos, st0["curr_target_index"], st0["swing_leg"])
    world = dict(phys)
    world["env_origins"] = sc.env_origins
    world["joint_pos_limits"] = sc.joint_limits.unsqueeze(0).repeat(num_envs, 1, 1)
    ref = rf.make_reference_env(world, sc.cfg, BODY_NAMES, JOINT_NAMES, su)
    assert torch.equal(ref.steps_pos, orc.steps_pos) and torch.equal(ref.steps_dphi, orc.steps_dphi)
    install_mdp_state(ref, st0, num_steps=S)
    install_mdp_state(orc, st0, num_steps=S)
    for step in range(12):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        rf.load_physics(ref, phys)
        r = rf.step_mdp(ref, phys["actions"], rf.UniformTables(m, n, sc.stone_uniforms(step)))
        o = orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(step))
        for a, b, what in zip(r, o, ("obs", "reward", "terminated", "time_out", "reset ids")):
            assert torch.equal(a, b), f"S={S} step {step}: {what}"
        for k in ("curr_target_index", "prev_target_index", "next_target_index", "swing_leg", "target_reach_count",
                  "episode_length_buf", "curriculum", "potentials", "steps_pos", "steps_dphi"):
            assert torch.equal(getattr(ref, k), getattr(orc, k)), f"S={S} step {step}: {k}"
