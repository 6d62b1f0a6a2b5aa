"""Test infrastructure: the oracle port driven the way the 3-call path (`pass1` -> `reset` -> `pass2`) draws.

`ThreeCallOracle` subclasses `AllstepsOracle` and differs from it in three ways:
* the grid curriculum and every draw of a reset use the handle's Philox step counter as the 3-call path leaves it --
  advanced by pass 1 before the reset of a step, and by the reset itself when it comes outside a step -- so in a run
  without such resets step k draws at k + 1;
* the stone draws come from `Scenario.stone_uniforms` at that counter, the mirror / noise draws from
  `Scenario.reset_uniforms`;
* `reset_outside_step` is `DirectRLEnv.reset()`: every env resets, draws a new bin and new stones, but no episode ended,
  so nothing is recorded in the histograms (`ThreeCallGrid.assign`).
The oracle port itself is unchanged.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import allsteps_oracle as ao
from oracle import grid_curriculum as gc


class ThreeCallGrid(gc.GridCurriculum):
    """`GridCurriculum` plus the assign-only turnover of a reset outside a step."""

    record = True  # False while a reset outside a step runs

    def assign(self, env_ids: np.ndarray, seed: int, step: int) -> np.ndarray:
        """New bins from the histograms as they stand; the histograms stay as they are."""
        cdf = gc.cdf_of(self.attempts, self.successes)
        self.bins[env_ids] = gc.sample_bins(cdf, gc.grid_draws(seed, step, env_ids + self.env_id_offset))
        return self.bins[env_ids]

    def episode_end(self, env_ids, index_at_end, num_stones, seed, step):
        if not self.record:
            return self.assign(env_ids, seed, step)
        return super().episode_end(env_ids, index_at_end, num_stones, seed, step)


class ThreeCallOracle(ao.AllstepsOracle):
    def __init__(self, sc, grid_bins: int = 0, intended_regen: bool = False):
        grid = ThreeCallGrid(sc.N, grid_bins, sc.env_id_offset) if grid_bins else None
        super().__init__(sc.cfg, sc.N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0),
                         intended_regen=intended_regen, grid=grid, seed=sc.seed)
        self.sc = sc
        self.counter = 0  # the handle's Philox step counter (a fresh handle generates its stones at 0)

    def _advance(self):
        self.counter += 1
        self.step_index = self.counter  # (AllstepsOracle draws the grid turnover at step_index)
        m, n = self.sc.reset_uniforms(self.counter)
        return m, n, self.sc.stone_uniforms(self.counter)

    def step(self, phys, actions):
        m, n, su = self._advance()
        return super().step(phys, actions, m, n, su)

    def reset_outside_step(self, phys):
        """`_reset_idx(all envs)` with no pass before it, then the observations (DRL:256-279)."""
        m, n, su = self._advance()
        self.load_physics(phys)
        if self.grid is not None:
            self.grid.record = False
        try:
            self.reset_rows(torch.arange(self.N), m, n, su)
        finally:
            if self.grid is not None:
                self.grid.record = True
        return self.observations()
