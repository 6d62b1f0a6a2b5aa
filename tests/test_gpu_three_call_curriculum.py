"""GPU: the difficulty-grid curriculum and stone regeneration on the 3-call path (`pass1` -> `reset` -> `pass2`, what
the DirectRLEnv hooks and the manager terms drive), against `ThreeCallOracle`, and the stone writes of both faces."""
from __future__ import annotations

import types

import numpy as np
import pytest
import torch

from scenario import Scenario, install_mdp_state
from test_gpu_faces import _Scene, _fake_world, _install
from test_gpu_memory_safety import guarded_buffers, guarded_mdp
from test_gpu_parity import close, close_obs, exact, to_views
from three_call_oracle import ThreeCallOracle

pytestmark = pytest.mark.gpu

STATE_KEYS = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")


def _physx_writes(keep, ids, out, k):
    """What the three robot writes of `_reset_idx` (ART:316-489) and scene.reset do to the data views."""
    keep["root_pos_w"][ids] = out.reset_root_state[:k, 0:3]
    keep["root_quat_w"][ids] = out.reset_root_state[:k, 3:7]
    keep["root_lin_vel_w"][ids] = out.reset_root_state[:k, 7:10]
    keep["joint_pos"][ids] = out.reset_joint_pos[:k]
    keep["joint_vel"][ids] = out.reset_joint_vel[:k]
    keep["force_matrix_right"][ids] = 0.0
    keep["force_matrix_left"][ids] = 0.0


def _grid_of(grid):
    return (torch.from_numpy(grid.bins.copy()), torch.from_numpy(grid.attempts.astype(np.int64)),
            torch.from_numpy(grid.successes.astype(np.int64)))


def run_three_call(N, steps, seed, grid_bins=0, intended_regen=False, device_list=False, fall=0.05,
                   high_index=False):
    """pass1 / reset / pass2 against ThreeCallOracle; every step compares masks, reward, obs, reset rows, state,
    stones, n_regenerated and (grid) bins and histograms.  Returns totals."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers

    sc = Scenario(N, seed=seed, fall_fraction=fall)
    st0 = sc.initial_mdp_state()
    if high_index:
        st0["curr_target_index"] = torch.randint(9, 20, (N,), generator=sc.gen)
    orc = ThreeCallOracle(sc, grid_bins=grid_bins, intended_regen=intended_regen)
    mdp = AllstepsMDP(N, device="cuda:0", seed=seed, grid_bins=grid_bins, intended_regen=intended_regen)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in STATE_KEYS})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    ep_len = st0["episode_length_buf"].cuda()
    totals = dict(resets=0, regen=0, quiet=0, busy=0)
    for step in range(steps):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        hist_before = mdp.grid_hist_tensor.clone()
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        views, keep = to_views(phys, origins, sc.body_indices)
        ep_len += 1  # DRL:351
        mdp.pass1(views, keep["actions"], out, episode_length=ep_len)
        order = None
        if device_list:
            mdp.reset(origins, None, out, episode_length=ep_len)
            n = int(out.n_reset.item())  # (the test plays PhysX: it needs the ids on the host side)
            ids = out.reset_ids[:n].long()
            order = ids.argsort()
            _physx_writes(keep, ids, out, n)
            mdp.pass2(views, out)
            ids = ids[order]
        else:
            ids = out.dones.nonzero().squeeze(-1)  # DRL:359
            if len(ids):
                mdp.reset(origins, ids, out, episode_length=ep_len)
                _physx_writes(keep, ids, out, len(ids))
                mdp.pass2(views, out)
            else:
                mdp.no_reset()  # DRL:360
        torch.cuda.synchronize()
        what = f"step {step}"
        exact(out.terminated, o_term, f"{what} terminated")
        exact(out.time_out, o_to, f"{what} time_out")
        close(out.reward, o_rew, f"{what} reward")
        exact(ids, o_ids, f"{what} reset ids")
        close_obs(out.obs, o_obs, f"{what} obs")
        k = len(o_ids)
        if k:
            w = orc.reset_writes
            rows = torch.cat((out.reset_root_state[:k], out.reset_joint_pos[:k]), -1)
            if order is not None:  # (the device-side list is in the order pass 1 compacted it)
                rows = rows[order]
            close(rows[:, :13], torch.cat((w["root_pose"], w["root_velocity"]), -1), f"{what} root rows")
            close(rows[:, 13:], w["joint_pos"], f"{what} joint_pos rows")
        exact(ep_len, orc.episode_length_buf, f"{what} episode_length")
        st = mdp.export_state()
        for key in ("curr_target_index", "swing_leg", "target_reach_count", "curriculum"):
            exact(st[key], getattr(orc, key), f"{what} {key}")
        close(st["potentials"], orc.potentials, f"{what} potentials")
        close(st["steps_pos"], orc.steps_pos, f"{what} steps_pos")
        close(st["steps_dphi"], orc.steps_dphi, f"{what} steps_dphi")
        n_regen = len(orc.regenerated_ids) if k else 0
        assert mdp.read_stats()["n_regenerated"] == n_regen, f"{what} n_regenerated"
        if grid_bins:
            bins, att, succ = mdp.grid_state()
            o_bins, o_att, o_succ = _grid_of(orc.grid)
            exact(bins, o_bins, f"{what} bins")
            exact(att, o_att, f"{what} attempts histogram")
            exact(succ, o_succ, f"{what} successes histogram")
            if not k:
                assert torch.equal(mdp.grid_hist_tensor, hist_before), f"{what}: a quiet step changed the histograms"
        # from here on both sides use the same stones, so that fp noise in sin/cos cannot flip a later mask
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        totals["resets"] += k
        totals["regen"] += n_regen
        totals["quiet" if not k else "busy"] += 1
    return totals, orc, mdp


@pytest.mark.parametrize("device_list", [False, True])
@pytest.mark.parametrize("regen_mode,N,steps", [("1", 3000, 10), ("2", 3000, 10), ("0", 700, 300),
                                                ("0", (1 << 17) + 37, 3)])
def test_grid_curriculum_on_the_three_call_path(regen_mode, N, steps, device_list, monkeypatch):
    """Kernel (c) behind as_reset: outcome -> histogram (joined when k_pass2_commit closes the step), new bin from
    the CDF of the previous steps, stones at the bin's difficulty, window at index 1.  regen_mode: the shape of
    k_reset_rows (1 warp per env, 2 thread per env, 0 by batch size: 2^17 + 37 envs take the thread per env and the
    prepared step-kernel instantiations)."""
    monkeypatch.setenv("ALLSTEPS_REGEN_MODE", regen_mode)
    B = 11
    totals, orc, mdp = run_three_call(N, steps, seed=19, grid_bins=B, device_list=device_list)
    assert totals["resets"] > 0 and totals["regen"] == totals["resets"]
    assert int(orc.grid.attempts.sum()) == totals["resets"]
    if steps >= 300:
        assert totals["resets"] > 500
        assert len(np.unique(orc.grid.bins)) > 30  # the sampler spreads over the grid


@pytest.mark.parametrize("device_list", [False, True])
def test_quiet_three_call_steps_leave_the_histograms_alone(device_list):
    """Steps in which nothing resets (as_step_no_reset; with the device-side list an empty list, which
    k_pass2_commit reverts) record no outcome."""
    totals, orc, _ = run_three_call(48, 12, seed=13, grid_bins=7, device_list=device_list, fall=0.0)
    assert totals["quiet"] > 0


@pytest.mark.parametrize("device_list", [False, True])
def test_intended_regeneration_on_the_three_call_path(device_list):
    totals, _, _ = run_three_call(1536, 8, seed=9, intended_regen=True, device_list=device_list, high_index=True)
    assert totals["regen"] > 0


class _FakeSteps:
    """A `RigidObjectCollection` that records `write_object_pose_to_sim`."""

    def __init__(self):
        self.calls = []

    def write_object_pose_to_sim(self, pose, env_ids):
        self.calls.append((pose.clone(), torch.as_tensor(env_ids).clone()))


def _check_stone_write(call, mdp, ids, what):
    pose, got_ids = call
    exact(got_ids.cpu(), ids.cpu(), f"{what}: ids of the stone write")
    pos = mdp.export_state(("steps_pos",))["steps_pos"][ids.to(mdp.device)]
    exact(pose[..., :3], pos, f"{what}: stone positions")
    quat = torch.tensor([1.0, 0.0, 0.0, 0.0], device=pose.device).expand(len(ids), 20, 4)
    exact(pose[..., 3:], quat, f"{what}: stone orientations")


def test_standalone_env_reset_then_steps_with_the_grid():
    """`StandaloneAllstepsEnv(..., grid_bins=B).reset()` before any step: every env draws a bin and stones at it, the
    histograms stay zero; then steps through the hooks match the oracle and every step that resets writes the new
    stones of exactly its reset envs."""
    from allsteps_isaaclab_b200.env import StandaloneAllstepsEnv

    N, seed, B = 600, 31, 11
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.05)
    orc = ThreeCallOracle(sc, grid_bins=B)
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    robot, left, right = _fake_world(sc, phys)
    scene = types.SimpleNamespace(env_origins=sc.env_origins.cuda())
    env = StandaloneAllstepsEnv(robot, left, right, scene, "cuda:0", sc.cfg, seed=seed, grid_bins=B)
    close(env.steps_pos, orc.steps_pos, "stones of the fresh handle")
    env.steps = _FakeSteps()
    o_obs = orc.reset_outside_step(phys)
    _install(robot, left, right, phys)
    obs, _ = env.reset()
    torch.cuda.synchronize()
    close_obs(obs["policy"], o_obs, "obs of the reset")
    bins, att, succ = env.mdp.grid_state()
    exact(bins, _grid_of(orc.grid)[0], "bins drawn by the reset")
    assert int(att.sum()) == 0 and int(succ.sum()) == 0, "a reset outside a step recorded outcomes"
    assert len(torch.unique(bins)) > 30
    close(env.steps_pos, orc.steps_pos, "stones of the reset")
    assert len(env.steps.calls) == 1
    _check_stone_write(env.steps.calls[0], env.mdp, torch.arange(N, device="cuda"), "reset")
    env.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    busy = 0
    for step in range(8):
        env.steps.calls.clear()
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        _install(robot, left, right, phys)
        obs, rew, term, to, _ = env.post_physics_step(phys["actions"].cuda())
        torch.cuda.synchronize()
        exact(term, o_term, f"step {step} terminated")
        close(rew, o_rew, f"step {step} reward")
        close_obs(obs["policy"], o_obs, f"step {step} obs")
        exact(env.curr_target_index, orc.curr_target_index, f"step {step} curr_target_index")
        close(env.steps_pos, orc.steps_pos, f"step {step} stones")
        b, a, s = env.mdp.grid_state()
        o_b, o_a, o_s = _grid_of(orc.grid)
        exact(b, o_b, f"step {step} bins")
        exact(a, o_a, f"step {step} attempts")
        exact(s, o_s, f"step {step} successes")
        if len(o_ids):
            busy += 1
            assert len(env.steps.calls) == 1
            _check_stone_write(env.steps.calls[0], env.mdp, o_ids.cuda(), f"step {step}")
        else:
            assert not env.steps.calls
        env.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    assert busy > 0


@pytest.mark.parametrize("kw", [dict(), dict(grid_bins=11), dict(intended_regen=True)])
def test_hooks_write_the_stones_of_the_reset_envs(kw):
    """A few hundred steps through the hooks on the env's own synthetic physics: with regeneration, every step that
    resets writes the stones of its reset envs (rewritten unchanged where intended regeneration kept them); without,
    the stones are never written.  With the grid: non-zero histograms, more than 30 bins in use."""
    from allsteps_isaaclab_b200.env import StandaloneAllstepsEnv

    N, seed = 700, 43
    steps = 300 if kw.get("grid_bins") else 40
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.05)
    phys = sc.physics(torch.zeros(N, 20, 3), torch.ones(N, dtype=torch.int64), torch.zeros(N, dtype=torch.int64))
    robot, left, right = _fake_world(sc, phys)
    scene = types.SimpleNamespace(env_origins=sc.env_origins.cuda())
    env = StandaloneAllstepsEnv(robot, left, right, scene, "cuda:0", sc.cfg, seed=seed, **kw)
    env.steps = _FakeSteps()
    busy = 0
    for step in range(steps):
        env.steps.calls.clear()
        st = env.mdp.export_state(("steps_pos", "curr_target_index", "swing_leg"))
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        _install(robot, left, right, phys)
        _, _, term, to, _ = env.post_physics_step(phys["actions"].cuda())
        ids = (term | to).nonzero().squeeze(-1)
        if not kw:
            assert not env.steps.calls
        elif len(ids):
            busy += 1
            assert len(env.steps.calls) == 1, f"step {step}: {len(env.steps.calls)} stone writes"
            _check_stone_write(env.steps.calls[0], env.mdp, ids, f"step {step}")
        else:
            assert not env.steps.calls
    if kw:
        assert busy > 0
    if kw.get("grid_bins"):
        bins, att, succ = env.mdp.grid_state()
        assert int(att.sum()) > 0 and int(succ.sum()) > 0
        assert len(torch.unique(bins)) > 30


def test_manager_terms_with_the_grid():
    """`terms.binding(env, grid_bins=B)` before the managers: `reset_allsteps` writes the stones of the reset envs to
    the scene's `steps` collection; `allsteps_grid` equals what `grid_state()` gives and runs no MDP pass."""
    from allsteps_isaaclab_b200 import terms

    N, seed, B = 700, 23, 9
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.05)
    st0 = sc.initial_mdp_state()
    orc = ThreeCallOracle(sc, grid_bins=B)
    install_mdp_state(orc, st0)
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    robot, left, right = _fake_world(sc, phys)
    stones = _FakeSteps()
    scene = _Scene(robot=robot, foot_contacts_left=left, foot_contacts_right=right, steps=stones)
    scene.env_origins = sc.env_origins.cuda()
    env = types.SimpleNamespace(num_envs=N, device="cuda:0", scene=scene, common_step_counter=0,
                                episode_length_buf=st0["episode_length_buf"].cuda().clone(),
                                actions=torch.zeros(N, 21, device="cuda"), step_dt=4.0 / 240.0)
    b = terms.binding(env, seed=seed, grid_bins=B)
    launches = b.mdp.launch_count
    log = terms.allsteps_grid(env, None)
    assert b.mdp.launch_count == launches and b.mdp.read_stats()["step_counter"] == 0
    assert float(log["attempts"]) == 0.0 and float(log["bins_visited"]) == 0.0
    b.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi, **{k: st0[k] for k in STATE_KEYS
                                                                                      if k != "episode_length_buf"}})
    busy = 0
    for step in range(6):
        stones.calls.clear()
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        _install(robot, left, right, phys)
        env.actions = phys["actions"].cuda()
        env.episode_length_buf += 1
        env.common_step_counter += 1
        terminated = terms.allsteps_terminated(env)
        time_out = terms.allsteps_time_out(env)
        exact(terminated, o_term, f"step {step} terminated")
        close(terms.allsteps_total_reward(env), o_rew, f"step {step} reward")
        ids = (terminated | time_out).nonzero().squeeze(-1)
        if len(ids):
            busy += 1
            scene.reset(env, ids)
            env.episode_length_buf[ids] = 0
            terms.reset_allsteps(env, ids)
            assert len(stones.calls) == 1
            _check_stone_write(stones.calls[0], b.mdp, ids, f"step {step}")
        else:
            assert not stones.calls
        obs = torch.cat([t(env) for t in terms.OBSERVATION_TERMS], dim=-1)
        torch.cuda.synchronize()
        close_obs(obs, o_obs, f"step {step} obs")
        bins, att, succ = b.mdp.grid_state()
        exact(bins, _grid_of(orc.grid)[0], f"step {step} bins")
        log = terms.allsteps_grid(env, ids)
        assert all(v.dim() == 0 and v.device.type == "cuda" for v in log.values())
        total = int(att.sum())
        assert float(log["attempts"]) == total
        assert abs(float(log["success_rate"]) - int(succ.sum()) / max(total, 1)) < 1e-6
        assert float(log["bins_visited"]) == int((att > 0).sum())
        b.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    assert busy > 0 and float(log["attempts"]) > 0


def test_grid_histogram_view_is_the_handle_state():
    from allsteps_isaaclab_b200.mdp import AllstepsMDP

    mdp = AllstepsMDP(1000, device="cuda:0", seed=2, grid_bins=6)
    att = torch.arange(36, dtype=torch.int64) * 7 + 3
    succ = torch.arange(36, dtype=torch.int64) * 2
    mdp.set_grid_state(attempts=att, successes=succ)
    torch.cuda.synchronize()
    h = mdp.grid_hist_tensor.cpu().long()
    assert torch.equal(h[:36], att) and torch.equal(h[256:292], succ)
    assert int(h[36:256].abs().sum()) == 0


@pytest.mark.parametrize("kw", [dict(grid_bins=6), dict(intended_regen=True)])
def test_guard_bands_and_determinism_of_the_three_call_path(kw):
    """The 3-call path with regeneration on a guarded workspace, host and device-side lists and a reset outside a
    step: no write outside the buffers, and two runs give identical bits."""
    from allsteps_isaaclab_b200 import synthetic as syn
    from allsteps_isaaclab_b200.mdp import PhysicsViews

    N, seed = 2000, 5
    sc = Scenario(N, seed=seed, fall_fraction=0.1)
    origins = sc.env_origins.cuda()
    runs = []
    for _ in range(2):
        mdp, ws = guarded_mdp(N, seed, **kw)
        out, g = guarded_buffers(N, None, reward_terms=False)
        mdp.generate_stones(origins)
        sc0 = Scenario(N, seed=seed)
        st0 = sc0.initial_mdp_state()
        st0["curr_target_index"] = torch.randint(9, 20, (N,), generator=sc0.gen)
        mdp.import_state({k: st0[k] for k in STATE_KEYS})
        gen = torch.Generator(device="cuda").manual_seed(seed)
        ep = torch.zeros(N, dtype=torch.int64, device="cuda")
        mdp.reset(origins, torch.arange(N, device="cuda"), out, episode_length=ep)  # outside a step
        st = mdp.export_state()
        d = syn.random_physics_state(sc.cfg, st["steps_pos"], st["curr_target_index"], st["swing_leg"], gen)
        mdp.pass2(PhysicsViews.from_dict(d, origins), out)
        for step in range(6):
            st = mdp.export_state()
            d = syn.random_physics_state(sc.cfg, st["steps_pos"], st["curr_target_index"], st["swing_leg"], gen,
                                         fall_fraction=0.1)
            v = PhysicsViews.from_dict(d, origins)
            ep += 1
            mdp.pass1(v, d["actions"], out, episode_length=ep)
            if step % 2:
                mdp.reset(origins, None, out, episode_length=ep)
                mdp.pass2(v, out)
            else:
                ids = out.dones.nonzero().squeeze(-1)
                if len(ids):
                    mdp.reset(origins, ids, out, episode_length=ep)
                    mdp.pass2(v, out)
                else:
                    mdp.no_reset()
        torch.cuda.synchronize()
        assert ws.intact() and all(x.intact() for x in g.values())
        runs.append((out.obs.clone(), mdp.export_state(), mdp.grid_state() if kw.get("grid_bins") else None,
                     mdp.read_stats()))
    assert torch.equal(runs[0][0], runs[1][0])
    for k in runs[0][1]:
        assert torch.equal(runs[0][1][k], runs[1][1][k]), k
    if runs[0][2] is not None:
        for x, y in zip(runs[0][2], runs[1][2]):
            assert torch.equal(x, y)
        assert int(runs[0][2][1].sum()) > 0
    assert runs[0][3] == runs[1][3]


def test_resume_between_three_call_steps_with_the_grid():
    """state_dict() between two 3-call steps with the grid; a fresh handle that loads it continues bit for bit."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers

    N, seed, B = 3000, 41, 7
    sc = Scenario(N, seed=seed, fall_fraction=0.2)
    origins = sc.env_origins.cuda()

    def fresh():
        m = AllstepsMDP(N, device="cuda:0", seed=seed, grid_bins=B)
        m.generate_stones(origins)
        return m

    def physics_for(m):
        st = m.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        d = {k: v.cuda() for k, v in phys.items()}
        return PhysicsViews.from_dict(d, origins, sc.body_indices), d

    def three_call(m, v, d, out, ep):
        ep += 1
        m.pass1(v, d["actions"], out, episode_length=ep)
        ids = out.dones.nonzero().squeeze(-1)
        if len(ids):
            m.reset(origins, ids, out, episode_length=ep)
            _physx_writes(d, ids, out, len(ids))
            m.pass2(v, out)
        else:
            m.no_reset()

    mdp = fresh()
    out = StepBuffers(N, "cuda:0")
    ep = torch.zeros(N, dtype=torch.int64, device="cuda")
    for _ in range(5):
        v, d = physics_for(mdp)
        three_call(mdp, v, d, out, ep)
    ckpt = mdp.state_dict()
    ep_ckpt = ep.clone()
    tail = [physics_for(mdp)]
    record = []
    for i in range(6):
        v, d = tail[i]
        d_copy = {k: t.clone() for k, t in d.items()}
        three_call(mdp, v, d, out, ep)
        torch.cuda.synchronize()
        record.append(({k: getattr(out, k).clone() for k in ("obs", "reward", "terminated", "time_out")},
                       mdp.export_state(), mdp.grid_state()))
        tail[i] = (PhysicsViews.from_dict(d_copy, origins, sc.body_indices), d_copy)
        tail.append(physics_for(mdp))
    resumed = fresh()
    resumed.load_state_dict(ckpt)
    out2 = StepBuffers(N, "cuda:0")
    ep2 = ep_ckpt.clone()
    for i in range(6):
        v, d = tail[i]
        three_call(resumed, v, d, out2, ep2)
        torch.cuda.synchronize()
        outs, state, grid = record[i]
        for k, ref in outs.items():
            assert torch.equal(getattr(out2, k), ref), f"step {i}: {k} differs after the resume"
        st = resumed.export_state()
        for k, ref in state.items():
            assert torch.equal(st[k], ref), f"step {i}: state {k} differs after the resume"
        for x, y in zip(resumed.grid_state(), grid):
            assert torch.equal(x, y), f"step {i}: grid state differs after the resume"
    assert int(record[-1][2][1].sum()) > 0
