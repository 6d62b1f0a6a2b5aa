"""The specification of AsStepOut.reward_terms and of AsStats on top of the oracle port (test infrastructure).

`TermsOracle` records, per step, what the step kernels report besides obs / reward / masks: the ten reward terms of
ENV:350-375 in `REWARD_COLUMNS` order (costs positive) for every env, terminated ones included; the `fell`, `so_fast`
and `died` masks; the index advances of pass 1 and of pass 2; the regenerated ids; the float64 sum of the reward.  From
these it builds the `AsStats` record `read_stats()` must report once the step is closed.  The terms are recomputed
from the attributes `rewards()` leaves behind, with the port's own expressions; their total is not restated here (see
`signed_total`, which the CPU suite holds bit-identical to `rewards()`).
"""
from __future__ import annotations

import torch

from oracle import allsteps_oracle as ao

STAT_FIELDS = ("n_envs", "n_reset", "n_terminated", "n_time_out", "n_fell", "n_so_fast", "n_died", "n_advanced",
               "sum_target_index", "n_regenerated", "level", "step_counter", "n_missed")


class TermsOracle(ao.AllstepsOracle):
    """`AllstepsOracle` that keeps `terms` (N,10), the per-step masks and counters, and `stats` of the last step."""

    def dones(self):
        out = super().dones()
        self.advanced1 = self.advanced.clone()  # mdp_pass of pass 1 (ENV:452-457)
        self.level_of_step = int(self.curriculum.max())
        # what pass 2 overwrites when some env resets
        self.pass1_foot_contact = self.foot_contact.clone()
        self.pass1_target_reached = self.target_reached.clone()
        self.pass1_foot_dist = self.foot_to_target_dist_xy.clone()
        self.joint_pos_scaled_pass1 = self.joint_pos_scaled.clone()
        return out

    def rewards(self):
        reward = super().rewards()
        self.terms = self.reward_terms()
        self.final_obs = self.observations()
        return reward

    def reward_terms(self) -> torch.Tensor:
        """ENV:350-375, one column per term, costs positive: the operands of the sum in `rewards()`."""
        c = self.cfg
        p = self.phys
        rows = torch.arange(self.N)
        alive = torch.ones_like(self.torso_to_feet_height) * c.alive_reward_scale
        progress = self.potentials - self.old_potentials
        roll_bad = (self.roll > 0.4) | (self.roll < -0.4)
        pitch_bad = (self.pitch > 0.4) | (self.pitch < -0.2)
        roll_cost = torch.where(roll_bad, self.roll.abs(), torch.zeros_like(self.roll))
        pitch_cost = torch.where(pitch_bad, self.pitch.abs(), torch.zeros_like(self.pitch))
        speed = torch.linalg.vector_norm(p["root_lin_vel_w"], dim=-1)
        speed_cost = torch.where(speed > 1.6, speed - 1.6, torch.zeros_like(speed))
        action_cost = c.actions_cost_scale * torch.linalg.vector_norm(self.actions, dim=-1)
        energy_cost = c.energy_cost_scale * torch.sum(torch.abs(p["joint_vel"] * self.actions), dim=-1)
        limit_cost = torch.count_nonzero(torch.abs(self.joint_pos_scaled) > 0.99, dim=-1).float() \
            * c.joint_at_limit_cost_scale
        pays_step = self.target_reached & (self.target_reach_count == 1) & (self.curr_target_index < self.S - 1)
        dist = self.foot_to_target_dist_xy[rows, self.swing_leg]
        step_reward = torch.where(pays_step, 50 * torch.exp(-dist / 0.25), torch.zeros_like(dist))
        at_goal = (self.curr_target_index == self.S - 1) & (self.body_dist_to_target_xy < 0.15)
        bonus = torch.where(at_goal, torch.full_like(dist, 10.0), torch.zeros_like(dist))
        return torch.stack((alive, progress, roll_cost, pitch_cost, speed_cost, energy_cost, action_cost,
                            limit_cost, step_reward, bonus), dim=-1)

    def reset_rows(self, env_ids, mirror_u, noise_u, stone_uniforms=None):
        super().reset_rows(env_ids, mirror_u, noise_u, stone_uniforms)
        self.advanced2 = self.advanced.clone()  # mdp_pass of pass 2 (ENV:567)

    def step(self, phys, actions, mirror_u=None, noise_u=None, stone_uniforms=None):
        self.advanced2 = torch.zeros(self.N, dtype=torch.bool)  # no env reset: pass 2 does not run (DRL:360)
        self.regenerated_ids = torch.zeros(0, dtype=torch.int64)
        step_counter = self.step_index
        out = super().step(phys, actions, mirror_u, noise_u, stone_uniforms)
        _, reward, term, time_out, ids = out
        self.last_reward = reward
        self.reward_sum = float(reward.double().sum())
        missed = int(self.missed_step_pass1.sum()) if self.missed_step_height is not None else 0
        self.stats = {
            "n_envs": self.N,
            "n_reset": len(ids),
            "n_terminated": int(term.sum()),
            "n_time_out": int(time_out.sum()),
            "n_fell": int(self.fell.sum()),
            "n_so_fast": int(self.so_fast.sum()),
            "n_died": int(self.died.sum()),
            "n_advanced": int(self.advanced1.sum()) + int(self.advanced2.sum()),
            "sum_target_index": int(self.pass1["curr_target_index"].sum()),
            "n_regenerated": len(self.regenerated_ids),
            "level": self.level_of_step,
            "step_counter": step_counter,
            "n_missed": missed,
        }
        return out


def signed_total(terms: torch.Tensor) -> torch.Tensor:
    """The terms summed the way the reference sums them, left to right (ENV:377-394)."""
    t = terms.unbind(-1)
    return t[0] + t[1] - t[2] - t[3] - t[4] - t[5] - t[6] - t[7] + t[8] + t[9]
