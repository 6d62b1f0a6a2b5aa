"""CPU, where the reference checkout is mounted: the oracle port's final observation (FinalObsOracle.final_obs, the
specification of AsStepOut.final_obs) against the reference's own `_get_observations()` called between `_get_dones` /
`_get_rewards` and `_reset_idx` of the same step."""
from __future__ import annotations

import pytest
import torch

from oracle import ref_loader

pytestmark = pytest.mark.skipif(not ref_loader.reference_available(), reason="reference checkout not mounted")


def test_port_final_obs_is_bit_identical_to_live_reference():
    from allsteps_isaaclab_b200.config import BODY_NAMES, JOINT_NAMES
    from final_obs_oracle import FinalObsOracle, record_reference_final_obs
    from oracle import ref_fake_env as rf
    from scenario import Scenario, install_mdp_state

    num_envs, steps = 64, 25
    sc = Scenario(num_envs, seed=31 + num_envs, full_bodies=True)
    su = sc.stone_uniforms(0)
    st0 = sc.initial_mdp_state()
    st0["episode_length_buf"][::9] = 897  # time-outs as well as terminations
    orc = FinalObsOracle(sc.cfg, num_envs, sc.env_origins, sc.joint_limits, sc.body_indices, su)
    phys = sc.physics(orc.steps_pos, st0["curr_target_index"], st0["swing_leg"])
    world = dict(phys)
    world["env_origins"] = sc.env_origins
    world["joint_pos_limits"] = sc.joint_limits.unsqueeze(0).repeat(num_envs, 1, 1)
    ref = rf.make_reference_env(world, sc.cfg, BODY_NAMES, JOINT_NAMES, su)
    record_reference_final_obs(ref)
    install_mdp_state(ref, st0)
    install_mdp_state(orc, st0)
    n_reset = n_time_out = 0
    for step in range(steps):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        rf.load_physics(ref, phys)
        r = rf.step_mdp(ref, phys["actions"], rf.UniformTables(m, n, sc.stone_uniforms(step)))
        o = orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(step))
        for a, b, what in zip(r, o, ("obs", "reward", "terminated", "time_out", "reset ids")):
            assert torch.equal(a, b), f"step {step}: {what}"
        assert torch.equal(ref.final_obs, orc.final_obs), f"step {step}: final_obs"
        n_reset += len(o[4])
        n_time_out += int(o[3].sum())
    assert n_reset > 0 and n_time_out > 0
