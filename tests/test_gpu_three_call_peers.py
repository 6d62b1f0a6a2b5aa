"""GPU: the global 3-call mode (`connect_self(three_call=True)`, `as_peer_three_call`) in one process.

A handle in the mode runs the same 3-call steps as a plain handle from the same state: its exchange behind pass 1
decides the promotion and "did any env reset", and adds the previous step's grid outcomes to the histograms.  With a
world of one that is the plain handle's arithmetic, moved: outputs, reset rows, final observations, state, levels and
bins must be bit-identical at every step, the histograms equal right after each pass 1 (between steps the mode's lag
one step behind), and the plain handle must agree with `ThreeCallOracle`.  The cross-shard half is
tests/test_gpu_multi_three_call.py."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from scenario import Scenario, install_mdp_state
from test_gpu_parity import close, close_obs, exact, to_views
from three_call_driver import assert_same_step, reset_rows, three_call_step
from three_call_oracle import ThreeCallOracle

pytestmark = pytest.mark.gpu

STATE_KEYS = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")


@pytest.mark.parametrize("device_list", [False, True])
@pytest.mark.parametrize("regen_mode", ["1", "2"])
@pytest.mark.parametrize("B", [5, 11])
def test_global_three_call_mode_equals_the_plain_path(B, regen_mode, device_list, monkeypatch):
    """36 steps of 96 envs with indices preloaded high (promotions) and every fourth step without falls (quiet steps);
    regen_mode: the shape of k_reset_rows (1 a warp per env, 2 a thread per env)."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers

    monkeypatch.setenv("ALLSTEPS_REGEN_MODE", regen_mode)
    N, seed, steps = 96, 61 + B, 36
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    st0["curr_target_index"] = torch.randint(9, 20, (N,), generator=sc.gen)
    st0["episode_length_buf"] = torch.randint(0, 600, (N,), generator=sc.gen)  # no time-outs: quiet steps stay quiet
    orc = ThreeCallOracle(sc, grid_bins=B)
    install_mdp_state(orc, st0)
    origins = sc.env_origins.cuda()
    mdps = [AllstepsMDP(N, device="cuda:0", seed=seed, grid_bins=B) for _ in range(2)]
    plain, glob = mdps
    glob.connect_self(three_call=True)
    for m in mdps:
        m.generate_stones(origins)
        m.import_state({k: st0[k] for k in STATE_KEYS})
        m.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    outs = [StepBuffers(N, "cuda:0", final_obs=True) for _ in mdps]
    eps = [st0["episode_length_buf"].cuda() for _ in mdps]
    quiet = busy = 0
    for step in range(steps):
        what = f"step {step}"
        sc.fall_fraction = 0.0 if step % 4 == 3 else 0.04
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        after = {}
        res = []
        for i, (m, out, ep) in enumerate(zip(mdps, outs, eps)):
            views, keep = to_views(phys, origins, sc.body_indices)

            def snap(i=i, m=m):
                torch.cuda.synchronize()
                after[i] = m.grid_hist_tensor.clone()

            res.append(three_call_step(m, views, keep, out, origins, ep, device_list, after_pass1=snap))
        torch.cuda.synchronize()
        (ids, order), (ids_g, order_g) = res
        assert torch.equal(after[0], after[1]), f"{what}: histograms differ right after pass 1"
        assert torch.equal(glob.grid_hist_tensor, after[1]), f"{what}: the mode's histograms changed after pass 1"
        exact(ids, o_ids, f"{what} reset ids")
        assert torch.equal(ids, ids_g), f"{what}: reset ids differ"
        assert_same_step((plain, outs[0]), (glob, outs[1]), what, reset_rows(outs[0], order),
                         reset_rows(outs[1], order_g))
        assert torch.equal(eps[0], eps[1])
        # the plain handle against the oracle
        exact(outs[0].terminated, o_term, f"{what} terminated")
        exact(outs[0].time_out, o_to, f"{what} time_out")
        close(outs[0].reward, o_rew, f"{what} reward")
        close_obs(outs[0].obs, o_obs, f"{what} obs")
        exact(eps[0], orc.episode_length_buf, f"{what} episode_length")
        st = plain.export_state()
        for key in ("curr_target_index", "swing_leg", "target_reach_count", "curriculum"):
            exact(st[key], getattr(orc, key), f"{what} {key}")
        close(st["steps_pos"], orc.steps_pos, f"{what} steps_pos")
        bins, att, succ = plain.grid_state()
        exact(bins, torch.from_numpy(orc.grid.bins.copy()), f"{what} bins")
        exact(att, torch.from_numpy(orc.grid.attempts.astype(np.int64)), f"{what} attempts")
        exact(succ, torch.from_numpy(orc.grid.successes.astype(np.int64)), f"{what} successes")
        # (both handles take the oracle's stones, so that fp noise in sin/cos cannot flip a later mask)
        for m in mdps:
            m.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        quiet += len(o_ids) == 0
        busy += len(o_ids) > 0
    assert quiet > 0 and busy > 0, (quiet, busy)
    assert int(orc.curriculum.max()) > 0, "no promotion happened; the test would prove nothing"
    s_plain, s_glob = plain.read_stats(), glob.read_stats()
    assert s_plain == s_glob, (s_plain, s_glob)


def test_misuse_of_the_global_three_call_mode():
    from allsteps_isaaclab_b200 import _cabi
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers

    N, seed = 256, 3
    mdp = AllstepsMDP(N, device="cuda:0", seed=seed)
    assert mdp.lib.as_peer_three_call(mdp.handle, 1) == -3, "the mode needs connected peers"
    assert b"as_peer_connect" in mdp.lib.as_last_error()
    mdp.connect_self(three_call=True)
    sc = Scenario(N, seed=seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    st = mdp.export_state()
    d = {k: v.cuda() for k, v in sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(),
                                            st["swing_leg"].cpu()).items()}
    views = PhysicsViews.from_dict(d, origins, sc.body_indices)
    out = StepBuffers(N, "cuda:0")
    with pytest.raises(_cabi.AllstepsLibraryError, match=r"\(-3\).*3-call mode"):
        mdp.step(views, d["actions"], out)
    mdp.pass1(views, d["actions"], out)
    assert mdp.lib.as_peer_three_call(mdp.handle, 0) == -3, "the mode is switched between steps only"
    mdp.no_reset()
    mdp.set_peer_three_call(False)
    mdp.step(views, d["actions"], out)  # (out of the mode the fused step runs again)
    torch.cuda.synchronize()


def test_resume_with_pending_grid_outcomes():
    """state_dict() between two steps of the mode, while the last step's grid outcomes are still pending; a fresh
    connected handle that loads it continues bit for bit -- outputs, state, bins and histograms."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers

    N, seed, B = 3000, 47, 7
    sc = Scenario(N, seed=seed, fall_fraction=0.2)
    origins = sc.env_origins.cuda()

    def fresh():
        m = AllstepsMDP(N, device="cuda:0", seed=seed, grid_bins=B)
        m.connect_self(three_call=True)
        m.generate_stones(origins)
        return m

    def physics_for(m):
        st = m.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        d = {k: v.cuda() for k, v in phys.items()}
        return PhysicsViews.from_dict(d, origins, sc.body_indices), d

    mdp = fresh()
    out = StepBuffers(N, "cuda:0")
    ep = torch.zeros(N, dtype=torch.int64, device="cuda")
    for i in range(5):
        v, d = physics_for(mdp)
        three_call_step(mdp, v, d, out, origins, ep, device_list=bool(i % 2))
    torch.cuda.synchronize()
    pending = mdp.exchange_tensor[mdp.grid_words].clone()
    assert int(pending.view(torch.int32).sum()) > 0, "no outcome is pending; the test would prove nothing"
    ckpt = mdp.state_dict()
    ep_ckpt = ep.clone()
    tail = [physics_for(mdp)]
    record = []
    for i in range(6):
        v, d = tail[i]
        d_copy = {k: t.clone() for k, t in d.items()}
        three_call_step(mdp, v, d, out, origins, ep, device_list=bool(i % 2))
        torch.cuda.synchronize()
        record.append(({k: getattr(out, k).clone() for k in ("obs", "reward", "terminated", "time_out")},
                       mdp.export_state(), mdp.grid_state()))
        tail[i] = (PhysicsViews.from_dict(d_copy, origins, sc.body_indices), d_copy)
        tail.append(physics_for(mdp))
    resumed = fresh()
    resumed.load_state_dict(ckpt)
    torch.cuda.synchronize()
    assert torch.equal(resumed.exchange_tensor[resumed.grid_words], pending), "pending outcomes were not restored"
    out2 = StepBuffers(N, "cuda:0")
    ep2 = ep_ckpt.clone()
    for i in range(6):
        v, d = tail[i]
        three_call_step(resumed, v, d, out2, origins, ep2, device_list=bool(i % 2))
        torch.cuda.synchronize()
        outs, state, grid = record[i]
        for k, ref in outs.items():
            assert torch.equal(getattr(out2, k), ref), f"step {i}: {k} differs after the resume"
        st = resumed.export_state()
        for k, ref in state.items():
            assert torch.equal(st[k], ref), f"step {i}: state {k} differs after the resume"
        for x, y in zip(resumed.grid_state(), grid):
            assert torch.equal(x, y), f"step {i}: grid state differs after the resume"
