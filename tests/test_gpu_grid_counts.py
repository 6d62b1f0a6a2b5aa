"""GPU: the difficulty-grid curriculum at the histogram counts of a long run, against the oracle
(oracle/grid_curriculum.py) on all three routes that close a step -- the fused step, the 3-call path (host id list and
device-side list) and the fused step closed on a handed-in global record.  The counts are preloaded with
`set_grid_state`: bins from 2^27 to 2^32 - 1 attempts, where a 64-bit weight numerator wraps, and bins right at the
top of the uint32 counters, where the fold halves them.  Also the Python faces of those counters."""
from __future__ import annotations

import types

import numpy as np
import pytest
import torch

from grid_counts import (SAMPLING_ENVS, SAMPLING_FALL, SAMPLING_GRIDS, SAMPLING_SEED, U32_MAX, at_the_top,
                         crafted_histograms)
from scenario import Scenario, install_mdp_state
from test_gpu_parity import close, exact, to_views
from test_gpu_three_call_curriculum import _physx_writes
from three_call_oracle import ThreeCallOracle

pytestmark = pytest.mark.gpu

STATE_KEYS = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")
ROUTES = ("fused", "three_call_host_ids", "three_call_device_list")


class _Run:
    """One handle and its oracle on the same scenario, stepped through one route; the grid is checked every step."""

    def __init__(self, route, N, B, seed, fall):
        from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers
        from oracle import allsteps_oracle as ao
        from oracle import grid_curriculum as gc

        self.route, self.N, self.B = route, N, B
        self.sc = sc = Scenario(N, seed=seed, fall_fraction=fall)
        st0 = sc.initial_mdp_state()
        if route.startswith("three_call"):
            self.orc = ThreeCallOracle(sc, grid_bins=B)
        else:
            self.orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices,
                                         sc.stone_uniforms(0), grid=gc.GridCurriculum(N, B), seed=seed)
        self.grid = self.orc.grid
        self.mdp = AllstepsMDP(N, device="cuda:0", seed=seed, grid_bins=B)
        self.origins = sc.env_origins.cuda()
        self.mdp.generate_stones(self.origins)
        install_mdp_state(self.orc, st0)
        self.mdp.import_state({k: st0[k] for k in STATE_KEYS})
        self.mdp.import_state({"steps_pos": self.orc.steps_pos, "steps_dphi": self.orc.steps_dphi})
        self.ep_len = st0["episode_length_buf"].cuda()
        self.out = StepBuffers(N, "cuda:0")
        self.step_no = 0
        self.resets = 0

    def set_grid(self, bins=None, att=None, succ=None):
        """The same grid state into the oracle and the handle."""
        if bins is not None:
            self.grid.bins[:] = bins
        if att is not None:
            self.grid.attempts[:] = att
            self.grid.successes[:] = succ
        self.mdp.set_grid_state(None if bins is None else torch.from_numpy(bins.astype(np.int64)),
                                None if att is None else torch.from_numpy(att.astype(np.int64)),
                                None if succ is None else torch.from_numpy(succ.astype(np.int64)))

    def step(self, before_fold=None):
        """One step on both sides.  before_fold(d_att) -> (att, succ): histograms to put in place once the step's
        per-bin outcomes are known (the oracle's turnover reads them; nothing before it does), on both sides."""
        orc, mdp, out, sc = self.orc, self.mdp, self.out, self.sc
        if before_fold is not None:
            grid, nb, preload = self.grid, self.B * self.B, {}
            turnover = grid.episode_end

            def hooked(env_ids, index_at_end, num_stones, seed, step):
                del grid.episode_end  # (one step only: back to the class method)
                att, succ = before_fold(np.bincount(grid.bins[env_ids], minlength=nb))
                grid.attempts[:], grid.successes[:] = att, succ
                preload.update(att=att.copy(), succ=succ.copy())
                return turnover(env_ids, index_at_end, num_stones, seed, step)

            grid.episode_end = hooked
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        if self.route.startswith("three_call"):
            o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        else:
            m, n = sc.reset_uniforms(self.step_no)
            o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(self.step_no))
        hist_before = None
        if before_fold is not None:
            assert preload, "no env ended an episode: the step folds nothing"
            hist_before = (preload["att"], preload["succ"])
            mdp.set_grid_state(attempts=torch.from_numpy(preload["att"].astype(np.int64)),
                               successes=torch.from_numpy(preload["succ"].astype(np.int64)))
        views, keep = to_views(phys, self.origins, sc.body_indices)
        if self.route == "fused":
            mdp.step(views, keep["actions"], out)
        elif self.route == "fused_global":  # as_fold_stats -> (the sum over the shards: one shard here) -> finish
            mdp.step(views, keep["actions"], out, finish=False)
            mdp.fold_stats()
            g = mdp.exchange_tensor.clone()
            mdp.finish_step(g)
        else:
            self.ep_len += 1
            mdp.pass1(views, keep["actions"], out, episode_length=self.ep_len)
            if self.route == "three_call_device_list":
                mdp.reset(self.origins, None, out, episode_length=self.ep_len)
                n = int(out.n_reset.item())
                ids = out.reset_ids[:n].long()
                _physx_writes(keep, ids, out, n)
                mdp.pass2(views, out)
            else:
                ids = out.dones.nonzero().squeeze(-1)
                if len(ids):
                    mdp.reset(self.origins, ids, out, episode_length=self.ep_len)
                    _physx_writes(keep, ids, out, len(ids))
                    mdp.pass2(views, out)
                else:
                    mdp.no_reset()
        torch.cuda.synchronize()
        what = f"{self.route} B={self.B} step {self.step_no}"
        exact(out.terminated, o_term, f"{what} terminated")
        bins, att, succ = mdp.grid_state()
        exact(bins, torch.from_numpy(self.grid.bins.copy()), f"{what} bins")
        exact(att, torch.from_numpy(self.grid.attempts.astype(np.int64)), f"{what} attempts histogram")
        exact(succ, torch.from_numpy(self.grid.successes.astype(np.int64)), f"{what} successes histogram")
        close(mdp.export_state(("steps_pos",))["steps_pos"], orc.steps_pos, f"{what} regenerated stones")
        # from here on both sides use the same stones, so that fp noise in sin/cos cannot flip a later mask
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        self.step_no += 1
        self.resets += len(o_ids)
        return hist_before, (att.cpu().numpy(), succ.cpu().numpy())


@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("regen_mode", ["1", "2"])
@pytest.mark.parametrize("B", SAMPLING_GRIDS)
def test_sampling_and_regeneration_at_large_counts(B, regen_mode, route, monkeypatch):
    """k_reset_rows (regen_mode 1: a warp per env, 2: a thread per env) draws from histograms of 2^27 .. 2^32 - 1
    attempts.  B = 16: 256 bins, every thread of the CTA's scan holds one, bin 255 is the top of the uint8 bin."""
    monkeypatch.setenv("ALLSTEPS_REGEN_MODE", regen_mode)
    run = _Run(route, SAMPLING_ENVS, B, SAMPLING_SEED, SAMPLING_FALL)
    att, succ = crafted_histograms(B, SAMPLING_SEED + B)
    bins = np.random.default_rng(B).integers(0, B * B, SAMPLING_ENVS).astype(np.uint8)
    assert (bins == B * B - 1).any()  # (outcomes are recorded against the last bin too: 255 for B = 16)
    run.set_grid(bins=bins, att=att, succ=succ)
    for _ in range(2):
        run.step()
    assert run.resets > 2000


@pytest.mark.parametrize("route", ROUTES[:2] + ("fused_global",))
def test_fold_at_the_top_of_the_counters(route):
    """Each fold site -- k_fixup_finish (fused; and closed on a handed-in global record, as_fold_stats ->
    as_finish_step(global)) and k_pass2_commit (3-call) -- with every bin that has outcomes da - 1, da or da + 1 below
    2^32 - 1: halved exactly when a + da passes 2^32 - 1, bin by bin as the oracle does."""
    B = 11
    run = _Run(route, 3000, B, 31, 0.3)
    run.set_grid(bins=np.random.default_rng(1).integers(0, B * B, 3000).astype(np.uint8))
    (a0, s0), (a1, s1) = run.step(before_fold=lambda da: at_the_top(da, 7))
    a0, s0 = a0.astype(np.int64), s0.astype(np.int64)
    halved = a1 < a0
    assert halved.sum() > 5 and (~halved & (a1 > a0)).sum() > 5, "both sides of the threshold must be met"
    assert np.all(s1 <= a1) and np.all(a1 <= U32_MAX)
    run.step()  # and the step after samples from the folded histograms


def _counts(mdp):
    bins, att, succ = mdp.grid_state()
    return bins.cpu().clone(), att.cpu().clone(), succ.cpu().clone()


def test_python_faces_of_the_counters():
    """grid_state() and the allsteps_grid log term read the counters as uint32; set_grid_state() refuses what the
    kernels' precondition excludes, before the handle is touched."""
    from allsteps_isaaclab_b200 import terms
    from allsteps_isaaclab_b200.mdp import AllstepsMDP

    N, B = 500, 6
    nb = B * B
    mdp = AllstepsMDP(N, device="cuda:0", seed=3, grid_bins=B)
    att = torch.full((nb,), U32_MAX, dtype=torch.int64)
    att[1], att[2] = 1 << 31, 0
    succ = att // 2
    succ[3] = U32_MAX
    bins = torch.arange(N) % nb
    mdp.set_grid_state(bins, att, succ)
    got = _counts(mdp)
    exact(got[0], bins.to(torch.uint8), "bins")
    exact(got[1], att, "attempts round trip")
    exact(got[2], succ, "successes round trip")
    env = types.SimpleNamespace()
    setattr(env, terms._KEY, types.SimpleNamespace(mdp=mdp))
    log = terms.allsteps_grid(env, None)
    assert float(log["attempts"]) == pytest.approx(float(att.sum()), rel=1e-6) and float(log["attempts"]) > 0
    assert float(log["success_rate"]) == pytest.approx(float(succ.sum()) / float(att.sum()), rel=1e-6)
    assert float(log["bins_visited"]) == nb - 1
    before = _counts(mdp)
    bad_counts = [(att.clone().index_fill_(0, torch.tensor([4]), -1), succ),
                  (att.clone().index_fill_(0, torch.tensor([4]), 1 << 32), succ),
                  (att, succ.clone().index_fill_(0, torch.tensor([5]), -1)),
                  (att.clone().index_fill_(0, torch.tensor([1]), 7), succ.clone().index_fill_(0, torch.tensor([1]), 8)),
                  (att[:-1], succ[:-1]), (att, succ[:-1]), (att.view(B, B), succ.view(B, B))]
    for a, s in bad_counts:
        with pytest.raises(ValueError):
            mdp.set_grid_state(attempts=a, successes=s)
    for bad_bins in (torch.full((N,), nb), torch.full((N,), -1), torch.zeros(N - 1, dtype=torch.int64),
                     torch.full((N,), 256)):
        with pytest.raises(ValueError):
            mdp.set_grid_state(bins=bad_bins)
    with pytest.raises(ValueError):
        mdp.set_grid_state(bins=bins, attempts=att, successes=succ + 1)  # nothing of a refused call is applied
    with pytest.raises(ValueError):
        mdp.set_grid_state(attempts=att)
    after = _counts(mdp)
    for x, y, name in zip(before, after, ("bins", "attempts", "successes")):
        exact(y, x, f"{name} after the refused calls")


def test_snapshot_and_restore_near_the_top_continue_bit_identically():
    from allsteps_isaaclab_b200.mdp import PhysicsViews, StepBuffers

    N, B, seed = 3000, 11, 41
    nb = B * B
    run = _Run("fused", N, B, seed, 0.2)
    att = np.full(nb, U32_MAX - 3, dtype=np.uint32)  # any bin with four outcomes or more is halved
    succ = (att // 3).astype(np.uint32)
    run.set_grid(bins=np.random.default_rng(2).integers(0, nb, N).astype(np.uint8), att=att, succ=succ)
    mdp, sc, origins = run.mdp, run.sc, run.origins
    snap = mdp.snapshot(include_stones=True)
    out = StepBuffers(N, "cuda:0")
    inputs, record = [], []
    for _ in range(2):
        st = mdp.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        d = {k: v.cuda() for k, v in phys.items()}
        inputs.append(d)
        mdp.step(PhysicsViews.from_dict(d, origins, sc.body_indices), d["actions"], out)
        torch.cuda.synchronize()
        record.append((out.obs.clone(), mdp.export_state(), _counts(mdp)))
    assert (record[-1][2][1].numpy() < att.astype(np.int64)).any(), "no bin reached the top"
    mdp.restore(snap, include_stones=True)
    exact(_counts(mdp)[1], torch.from_numpy(att.astype(np.int64)), "attempts after the restore")
    for i, d in enumerate(inputs):
        mdp.step(PhysicsViews.from_dict(d, origins, sc.body_indices), d["actions"], out)
        torch.cuda.synchronize()
        assert torch.equal(out.obs, record[i][0]), f"step {i}: obs"
        st = mdp.export_state()
        for k, ref in record[i][1].items():
            assert torch.equal(st[k], ref), f"step {i}: state {k}"
        for x, y in zip(_counts(mdp), record[i][2]):
            assert torch.equal(x, y), f"step {i}: grid state"
