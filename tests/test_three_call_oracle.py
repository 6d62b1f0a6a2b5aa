"""CPU: the test-side oracle of the grid curriculum on the 3-call path (tests/three_call_oracle.py)."""
from __future__ import annotations

import numpy as np
import torch

from oracle import grid_curriculum as gc
from scenario import Scenario
from three_call_oracle import ThreeCallGrid, ThreeCallOracle


def _grown_grid(N, B, seed):
    g = ThreeCallGrid(N, B)
    rng = np.random.default_rng(seed)
    for step in range(5):  # some history, so that the CDF is not flat
        ids = np.sort(rng.choice(N, N // 3, replace=False))
        g.episode_end(ids, rng.integers(0, 20, ids.shape[0]), 20, seed, step)
    return g


def test_assign_draws_the_bins_of_episode_end_and_records_nothing():
    N, B, seed, step = 500, 7, 3, 11
    g = _grown_grid(N, B, seed)
    ref = ThreeCallGrid(N, B)
    ref.bins, ref.attempts, ref.successes = g.bins.copy(), g.attempts.copy(), g.successes.copy()
    ids = np.arange(0, N, 2)
    att, succ = g.attempts.copy(), g.successes.copy()
    assigned = g.assign(ids, seed, step).copy()
    assert np.array_equal(g.attempts, att) and np.array_equal(g.successes, succ)
    drawn = ref.episode_end(ids, np.full(ids.shape[0], 15), 20, seed, step)
    assert np.array_equal(assigned, drawn)
    assert int(ref.attempts.sum()) == int(att.sum()) + ids.shape[0]
    assert len(np.unique(assigned)) > 5


def test_episode_end_with_recording_off_is_assign():
    N, B, seed = 300, 5, 8
    a, b = _grown_grid(N, B, seed), _grown_grid(N, B, seed)
    ids = np.arange(N)
    b.record = False
    drawn = b.episode_end(ids, np.full(N, 19), 20, seed, 4)
    assert np.array_equal(drawn, a.assign(ids, seed, 4))
    assert np.array_equal(b.attempts, a.attempts) and np.array_equal(b.successes, a.successes)


def test_reset_outside_a_step_assigns_bins_and_regenerates_at_the_next_counter():
    N, B = 200, 11
    sc = Scenario(N, seed=5)
    orc = ThreeCallOracle(sc, grid_bins=B)
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    orc.reset_outside_step(phys)
    assert orc.counter == 1
    assert int(orc.grid.attempts.sum()) == 0 and int(orc.grid.successes.sum()) == 0
    u24 = gc.grid_draws(sc.seed, 1, np.arange(N))
    expect = gc.sample_bins(gc.cdf_of(orc.grid.attempts, orc.grid.successes), u24)
    assert np.array_equal(orc.grid.bins, expect)
    pos, _ = gc.generate_stones_for_bins(sc.cfg, torch.from_numpy(expect), B, sc.stone_uniforms(1))
    assert torch.equal(orc.steps_pos, pos + sc.env_origins.unsqueeze(1))
    # a step after it records the outcomes of the envs that reset in it, drawing at counter 2
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    _, _, _, _, ids = orc.step(phys, phys["actions"])
    assert orc.counter == 2 and int(orc.grid.attempts.sum()) == len(ids)
