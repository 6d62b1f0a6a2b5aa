"""The specification of AsStepOut.final_obs on top of the oracle port and of the hosted reference (test infrastructure).

The final observation of env e in step t is the row `_get_observations()` (ENV:326-345) returns when it is called
between `_get_rewards()` and `_reset_idx()` of step t.  Both `AllstepsOracle.step` and `ref_fake_env.step_mdp` call the
rewards right before the reset, so the row is recorded at the end of that call; nothing else about the step changes.
"""
from __future__ import annotations

from oracle import allsteps_oracle as ao


class FinalObsOracle(ao.AllstepsOracle):
    """`AllstepsOracle` that keeps `final_obs` (N,59) of the last step: `observations()` on the pass-1 state."""

    def rewards(self):
        reward = super().rewards()
        self.final_obs = self.observations()
        return reward


def record_reference_final_obs(env):
    """Make the hosted reference env keep `env.final_obs`: its own `_get_observations()` right after `_get_rewards()`."""
    get_rewards = env._get_rewards

    def _get_rewards():
        reward = get_rewards()
        env.final_obs = env._get_observations()["policy"].clone()
        return reward

    env._get_rewards = _get_rewards
