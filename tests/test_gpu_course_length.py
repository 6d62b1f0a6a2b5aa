"""GPU: courses of 3 to 32 stones (`AllstepsCfg.num_steps`) through every layer -- fused step and 3-call path against
the oracle port, stone generation and regeneration in both kernel shapes, the last stone in pass 1 and pass 2, state
exchange, checkpoints, guard bands, the Isaac Lab faces -- and S = 20 as a control that must be bit-identical to a
handle created with num_steps = 0 (the default of a zero-initialised AsParams) and launch the same kernels.

Bar as in test_gpu_parity.py: masks, indices and counters bit-exact; fp32 within 1e-5 * max(1, |b|)."""
from __future__ import annotations

import re
import types

import pytest
import torch

from final_obs_oracle import FinalObsOracle
from scenario import Scenario, install_mdp_state
from test_gpu_faces import _fake_world, _install, _Scene
from test_gpu_memory_safety import Guarded, guarded_buffers
from test_gpu_parity import close, close_obs, exact, to_views
from test_gpu_three_call_curriculum import STATE_KEYS, _FakeSteps, _grid_of, _physx_writes
from three_call_oracle import ThreeCallOracle

pytestmark = pytest.mark.gpu

LENGTHS = (3, 4, 7, 12, 31, 32)


def cfg_of(S: int, **kw):
    from allsteps_isaaclab_b200.config import AllstepsCfg

    return AllstepsCfg(num_steps=S, **kw)


def make_mdp(S, N, seed, **kw):
    from allsteps_isaaclab_b200.mdp import AllstepsMDP

    return AllstepsMDP(N, device="cuda:0", seed=seed, cfg=kw.pop("cfg", None) or cfg_of(S), **kw)


def high_start(sc, S):
    """Mid-episode state with indices near the end of the course, so that envs reach the last stone."""
    st0 = sc.initial_mdp_state()
    st0["curr_target_index"] = torch.randint(max(S - 4, 1), S, (sc.N,), generator=sc.gen)
    return st0


def compare_state(mdp, orc, what, S):
    st = mdp.export_state()
    assert tuple(st["steps_pos"].shape) == (mdp.num_envs, S, 3) and tuple(st["steps_dphi"].shape) == (mdp.num_envs, S)
    for key in ("curr_target_index", "prev_target_index", "next_target_index", "swing_leg", "target_reach_count",
                "episode_length_buf", "curriculum"):
        exact(st[key], getattr(orc, key), f"{what} {key}")
    close(st["potentials"], orc.potentials, f"{what} potentials")
    close(st["steps_pos"], orc.steps_pos, f"{what} steps_pos")
    close(st["steps_dphi"], orc.steps_dphi, f"{what} steps_dphi")
    return st


def synthetic(sc, orc, step):
    return sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)


def run_fused(S, N, steps, seed, layout="contiguous", reward_terms=True, final_obs=True, intended_regen=False,
              missed_step=None, cfg=None, prepare=None, physics=synthetic):
    """Fused steps against the oracle; returns totals.  prepare(sc, st0) may edit the start state, physics(sc, orc,
    step) the physics of a step."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    cfg = cfg or cfg_of(S, **({} if missed_step is None else dict(missed_step_height=missed_step)))
    sc = Scenario(N, seed=seed, full_bodies=(layout == "isaac"), fall_fraction=0.05, cfg=cfg)
    st0 = high_start(sc, S)
    if prepare is not None:
        prepare(sc, st0)
    orc = FinalObsOracle(cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0),
                         intended_regen=intended_regen, missed_step_height=missed_step)
    mdp = make_mdp(S, N, seed, cfg=cfg, intended_regen=intended_regen, missed_step=missed_step is not None)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)  # in-kernel Philox at step counter 0, warp per env
    install_mdp_state(orc, st0, num_steps=S)
    mdp.import_state({k: st0[k] for k in STATE_KEYS})
    compare_state(mdp, orc, "initial", S)
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0", reward_terms=reward_terms, final_obs=final_obs)
    t = dict(resets=0, regen=0, last1=0, bonus=0, time_out=0, missed=0)
    for step in range(steps):
        phys = physics(sc, orc, step)
        before = orc.curr_target_index.clone()
        m, n = sc.reset_uniforms(step)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(step))
        views, keep = to_views(phys, origins, sc.body_indices, layout)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        what = f"S={S} N={N} step {step}"
        exact(out.terminated, o_term, f"{what} terminated")
        exact(out.time_out, o_to, f"{what} time_out")
        close(out.reward, o_rew, f"{what} reward")
        close_obs(out.obs, o_obs, f"{what} obs")
        n_reset = int(out.n_reset.item())
        ids = out.reset_ids[:n_reset].long().sort().values
        exact(ids, o_ids, f"{what} reset ids")
        idx1 = orc.pass1["curr_target_index"]
        if reward_terms:
            rt = out.reward_terms.cpu()
            alive = ~o_term
            total = rt[:, 0] + rt[:, 1] - rt[:, 2:8].sum(-1) + rt[:, 8] + rt[:, 9]
            close(total[alive], o_rew[alive], f"{what} reward terms", rtol=1e-4)
            at_end = (idx1 == S - 1) & (before == S - 1)
            assert bool((rt[at_end, 8] == 0).all()), f"{what}: a step reward was paid on the last stone"
            assert bool((rt[idx1 != S - 1, 9] == 0).all()), f"{what}: a bonus was paid before the last stone"
            t["bonus"] += int((rt[:, 9] == 10).sum())
        if final_obs and n_reset:
            close_obs(out.final_obs[ids], orc.final_obs[ids.cpu()], f"{what} final_obs")
        if n_reset:
            w = orc.reset_writes
            close(out.reset_root_state[ids], torch.cat((w["root_pose"], w["root_velocity"]), -1), f"{what} root rows")
            close(out.reset_joint_pos[ids], w["joint_pos"], f"{what} joint_pos rows")
        compare_state(mdp, orc, what, S)
        stats = mdp.read_stats()
        assert stats["n_reset"] == len(o_ids) and stats["sum_target_index"] == int(idx1.sum()), what
        regen = len(orc.regenerated_ids) if (intended_regen and n_reset) else 0
        assert stats["n_regenerated"] == regen, f"{what} n_regenerated"
        if missed_step is not None:
            assert stats["n_missed"] == int(orc.missed_step_pass1.sum()), f"{what} n_missed"
            t["missed"] += stats["n_missed"]
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        t["resets"] += n_reset
        t["regen"] += regen
        t["last1"] += int(((idx1 == S - 1) & (before == S - 2)).sum())
        t["time_out"] += int(o_to.sum())
    return t, mdp


def run_three_call(S, N, steps, seed, device_list, layout="contiguous", grid_bins=0, intended_regen=False,
                   outside_reset=False, cfg=None, prepare=None, physics=synthetic):
    """pass1 / reset / pass2 (or no_reset) against ThreeCallOracle; optionally a reset outside a step first."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    cfg = cfg or cfg_of(S)
    sc = Scenario(N, seed=seed, full_bodies=(layout == "isaac"), fall_fraction=0.05, cfg=cfg)
    st0 = high_start(sc, S)
    if prepare is not None:
        prepare(sc, st0)
    orc = ThreeCallOracle(sc, grid_bins=grid_bins, intended_regen=intended_regen)
    mdp = make_mdp(S, N, seed, cfg=cfg, grid_bins=grid_bins, intended_regen=intended_regen)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    compare_state(mdp, orc, "fresh handle", S)
    install_mdp_state(orc, st0, num_steps=S)
    mdp.import_state({k: st0[k] for k in STATE_KEYS})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    ep_len = st0["episode_length_buf"].cuda()
    if outside_reset:  # DirectRLEnv.reset(): `_reset_idx(all ids)` with no pass before it, then pass 2
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        o_obs = orc.reset_outside_step(phys)
        views, keep = to_views(phys, origins, sc.body_indices, layout)
        ids = torch.arange(N, device="cuda")
        mdp.reset(origins, ids, out, episode_length=ep_len)
        _physx_writes(keep, ids, out, N)
        mdp.pass2(views, out)
        torch.cuda.synchronize()
        close_obs(out.obs, o_obs, f"S={S} reset outside a step: obs")
        compare_state(mdp, orc, f"S={S} reset outside a step", S)
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    t = dict(resets=0, regen=0, last1=0, last2=0, busy=0)
    for step in range(steps):
        phys = physics(sc, orc, step)
        before = orc.curr_target_index.clone()
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        views, keep = to_views(phys, origins, sc.body_indices, layout)
        ep_len += 1
        mdp.pass1(views, keep["actions"], out, episode_length=ep_len)
        order = None
        if device_list:
            mdp.reset(origins, None, out, episode_length=ep_len)
            n = int(out.n_reset.item())
            ids = out.reset_ids[:n].long()
            order = ids.argsort()
            _physx_writes(keep, ids, out, n)
            mdp.pass2(views, out)
            ids = ids[order]
        else:
            ids = out.dones.nonzero().squeeze(-1)
            if len(ids):
                mdp.reset(origins, ids, out, episode_length=ep_len)
                _physx_writes(keep, ids, out, len(ids))
                mdp.pass2(views, out)
            else:
                mdp.no_reset()
        torch.cuda.synchronize()
        what = f"S={S} N={N} 3-call step {step}"
        exact(out.terminated, o_term, f"{what} terminated")
        exact(out.time_out, o_to, f"{what} time_out")
        close(out.reward, o_rew, f"{what} reward")
        exact(ids, o_ids, f"{what} reset ids")
        close_obs(out.obs, o_obs, f"{what} obs")
        k = len(o_ids)
        if k:
            w = orc.reset_writes
            rows = torch.cat((out.reset_root_state[:k], out.reset_joint_pos[:k]), -1)
            if order is not None:
                rows = rows[order]
            close(rows[:, :13], torch.cat((w["root_pose"], w["root_velocity"]), -1), f"{what} root rows")
            close(rows[:, 13:], w["joint_pos"], f"{what} joint_pos rows")
        exact(ep_len, orc.episode_length_buf, f"{what} episode_length")
        compare_state(mdp, orc, what, S)
        n_regen = len(orc.regenerated_ids) if k else 0
        assert mdp.read_stats()["n_regenerated"] == n_regen, f"{what} n_regenerated"
        if grid_bins:
            bins, att, succ = mdp.grid_state()
            o_bins, o_att, o_succ = _grid_of(orc.grid)
            exact(bins, o_bins, f"{what} bins")
            exact(att, o_att, f"{what} attempts")
            exact(succ, o_succ, f"{what} successes")
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        idx1 = orc.pass1["curr_target_index"]
        not_reset = torch.ones(N, dtype=torch.bool)
        not_reset[o_ids] = False
        t["resets"] += k
        t["regen"] += n_regen
        t["busy"] += int(k > 0)
        t["last1"] += int(((idx1 == S - 1) & (before == S - 2)).sum())
        t["last2"] += int(((orc.curr_target_index == S - 1) & (idx1 == S - 2) & not_reset).sum())
    return t, mdp


# ---------------------------------------------------------------------------------------------- the step paths
@pytest.mark.parametrize("S", LENGTHS + (20,))
@pytest.mark.parametrize("N,layout", [(64, "contiguous"), (1001, "contiguous"), (65580, "contiguous"),
                                      (65580, "isaac")])
def test_fused_step_against_the_oracle(S, N, layout):
    """N = 65 580 takes k_prepare* (the separate gather) and a ragged last tile; "isaac": (N,13) root and (N,17,13) body
    slices.  Defaults (no reward terms, no final_obs) where the FAST instantiations would be eligible at S = 20."""
    steps = 3 if N > 4096 else 8
    extras = N == 1001
    t, _ = run_fused(S, N, steps, seed=11 + S, layout=layout, reward_terms=extras, final_obs=extras)
    assert t["resets"] > 0


@pytest.mark.parametrize("S", LENGTHS + (20,))
@pytest.mark.parametrize("N,layout,device_list", [(64, "contiguous", False), (1001, "contiguous", True),
                                                  (65580, "contiguous", True), (65580, "isaac", False)])
def test_three_call_path_against_the_oracle(S, N, layout, device_list):
    steps = 3 if N > 4096 else 8
    t, _ = run_three_call(S, N, steps, seed=5 + S, device_list=device_list, layout=layout)
    assert t["resets"] > 0


def test_one_million_envs_at_32_stones():
    t, _ = run_fused(32, 1 << 20, 2, seed=3, reward_terms=False, final_obs=False)
    assert t["resets"] > 0


@pytest.mark.parametrize("S", (3, 12, 32))
@pytest.mark.parametrize("device_list", [False, True])
def test_reset_outside_a_step(S, device_list):
    run_three_call(S, 700, 3, seed=17, device_list=device_list, outside_reset=True)


# ---------------------------------------------------------------------------------------------- the last stone
def last_stone(S, stop_frames):
    """(prepare, physics) that place a third of the envs by hand: index S-2 (stop_frames 2) or S-3 (stop_frames 1), the
    right foot -- the swing leg -- pressing on the current stone, the left foot on the one after it, the root above the
    last stone; every 17th of them about to time out."""
    marked = {}

    def prepare(sc, st0):
        e = torch.arange(0, sc.N, 3)
        st0["curr_target_index"][e] = S - 4 + stop_frames
        st0["swing_leg"][e] = 0
        st0["target_reach_count"][e] = stop_frames - 1
        st0["episode_length_buf"][e[::17]] = sc.cfg.max_episode_length - 2
        marked["e"] = e

    def physics(sc, orc, step):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        e = marked["e"]
        idx = orc.curr_target_index[e]
        nxt = (idx + 1).clamp(max=S - 1)
        rf, lf = sc.body_indices[0], sc.body_indices[1]
        phys["body_pos_w"][e, rf, :2] = orc.steps_pos[e, idx, :2]
        phys["body_pos_w"][e, lf, :2] = orc.steps_pos[e, nxt, :2]
        phys["root_pos_w"][e, :2] = orc.steps_pos[e, S - 1, :2]
        for k in ("force_matrix_right", "force_matrix_left"):
            phys[k][e] = 0.0
        phys["force_matrix_right"][e, 0, idx, 2] = 150.0
        phys["force_matrix_left"][e, 0, nxt, 2] = 150.0
        return phys

    return prepare, physics


@pytest.mark.parametrize("S", LENGTHS + (20,))
def test_last_stone_in_pass_one_and_pass_two(S):
    """Envs driven from S-2 onto the last stone: in pass 1 (stop_frames 2: goal bonus, no step reward on the last stone,
    time-outs on the way), and in pass 2 (stop_frames 1: pass 1 moves S-3 -> S-2, pass 2 on the unchanged physics
    S-2 -> S-1), fused and 3-call, against the oracle."""
    prepare, physics = last_stone(S, 2)
    t, _ = run_fused(S, 1500, 3, seed=41, prepare=prepare, physics=physics)
    assert t["last1"] > 0 and t["bonus"] > 0 and t["time_out"] > 0
    t3, _ = run_three_call(S, 1500, 3, seed=41, device_list=True, prepare=prepare, physics=physics)
    assert t3["last1"] > 0
    prepare, physics = last_stone(S, 1)
    cfg1 = cfg_of(S, stop_frames=1)
    t, _ = run_fused(S, 1500, 2, seed=43, cfg=cfg1, prepare=prepare, physics=physics)
    t3, _ = run_three_call(S, 1500, 2, seed=43, device_list=False, cfg=cfg1, prepare=prepare, physics=physics)
    assert t3["last2"] > 0, "no env stepped onto the last stone in pass 2"


# ---------------------------------------------------------------------------------------------- stones
@pytest.mark.parametrize("regen_mode", ["1", "2"])
@pytest.mark.parametrize("S", (3, 7, 12, 32))
def test_regeneration_in_both_kernel_shapes(S, regen_mode, monkeypatch):
    """Intended regeneration (idx > S//2 at the end of the episode) on the fused and the 3-call path, and the grid
    curriculum with its success threshold at S//2, by the warp-per-env (1) and the thread-per-env (2) generator."""
    monkeypatch.setenv("ALLSTEPS_REGEN_MODE", regen_mode)
    t, _ = run_fused(S, 1500, 6, seed=23, intended_regen=True)
    assert t["regen"] > 0
    t, _ = run_three_call(S, 1500, 6, seed=29, device_list=True, intended_regen=True)
    assert t["regen"] > 0
    t, mdp = run_three_call(S, 1500, 6, seed=31, device_list=False, grid_bins=11)
    assert t["regen"] > 0 and int(mdp.grid_state()[2].sum()) > 0


@pytest.mark.parametrize("S", LENGTHS)
def test_generation_with_explicit_uniforms_and_philox(S):
    from oracle import allsteps_oracle as ao

    N = 777
    sc = Scenario(N, seed=8, cfg=cfg_of(S))
    mdp = make_mdp(S, N, 8)
    origins = sc.env_origins.cuda()
    u = torch.rand(5, N, S, generator=sc.gen)
    ref = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, u)
    mdp.generate_stones(origins, uniforms=u.cuda())
    st = mdp.export_state(("steps_pos", "steps_dphi"))
    close(st["steps_pos"], ref.steps_pos, "explicit uniforms steps_pos")
    close(st["steps_dphi"], ref.steps_dphi, "explicit uniforms steps_dphi")
    ids = torch.arange(0, N, 5)
    mdp.generate_stones(origins, env_ids=ids, uniforms=u[:3].contiguous().cuda())
    with pytest.raises(ValueError, match="num_steps"):
        mdp.generate_stones(origins, uniforms=torch.rand(5, N, 20 if S != 20 else 12, device="cuda"))
    ref = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    mdp.generate_stones(origins)
    close(mdp.export_state(("steps_pos",))["steps_pos"], ref.steps_pos, "philox steps_pos")


@pytest.mark.parametrize("S", (3, 12, 32))
def test_missed_step_termination(S):
    t, _ = run_fused(S, 1500, 5, seed=19, missed_step=0.12)  # (the synthetic swing foot hovers 0.11 m up)
    assert t["missed"] > 0


# ---------------------------------------------------------------------------------------------- state and checkpoints
@pytest.mark.parametrize("S", (3, 12, 32))
def test_export_import_stone_poses_snapshot_and_state_dict(S):
    from allsteps_isaaclab_b200.mdp import StepBuffers

    N = 999
    t, mdp = run_three_call(S, N, 2, seed=51, device_list=True)
    st = mdp.export_state()
    # stone poses in PhysX' object-major (S*N,7) layout
    poses, view_ids = mdp.export_stone_poses()
    assert tuple(poses.shape) == (S * N, 7) and tuple(view_ids.shape) == (S * N,)
    exact(poses.view(S, N, 7)[..., :3].permute(1, 0, 2), st["steps_pos"], "stone poses")
    exact(view_ids, torch.arange(S * N, dtype=torch.int32, device="cuda"), "view ids")
    ids = torch.tensor([5, 0, N - 1], device="cuda")
    buf = torch.full((S * N, 7), -7.0, device="cuda")
    _, vid = mdp.export_stone_poses(ids, buf)
    rows = (torch.arange(S, device="cuda")[:, None] * N + ids[None, :].int()).reshape(-1)
    exact(vid, rows.int(), "listed view ids")
    assert int((buf[:, 0] != -7.0).sum()) == 3 * S
    with pytest.raises(ValueError):
        mdp.export_stone_poses(view_poses=torch.zeros(20 * N if S != 20 else 12 * N, 7, device="cuda"))
    # export -> import round trip, with the index clamped to S-1
    mdp2 = make_mdp(S, N, 51)
    imp = dict(st)
    imp["curr_target_index"] = st["curr_target_index"].clone()
    imp["curr_target_index"][:7] = 40
    mdp2.import_state(imp)
    st2 = mdp2.export_state()
    exact(st2["curr_target_index"][:7], torch.full((7,), S - 1, device="cuda"), "clamped index")
    for k in ("steps_pos", "steps_dphi", "swing_leg", "potentials"):
        exact(st2[k], st[k], f"import {k}")
    with pytest.raises(ValueError):
        mdp2.import_state({"steps_pos": torch.zeros(N, 20 if S != 20 else 12, 3)})
    # snapshot / restore and state_dict: a resumed run is bit-identical
    ckpt = mdp.state_dict()
    assert int(ckpt["meta"][-1]) == S
    snap = mdp.snapshot()
    sc = Scenario(N, seed=52, cfg=cfg_of(S))
    origins = sc.env_origins.cuda()
    phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())

    def two_steps(m):
        out = StepBuffers(N, "cuda:0")
        res = []
        for _ in range(2):
            views, keep = to_views(phys, origins, sc.body_indices)
            m.step(views, keep["actions"], out)
            res.append((out.obs.clone(), out.reward.clone(), out.dones.clone()))
        return res, m.export_state()

    a, sa = two_steps(mdp)
    mdp.restore(snap)
    b, sb = two_steps(mdp)
    mdp3 = make_mdp(S, N, 51)
    mdp3.load_state_dict(ckpt)
    c, sc3 = two_steps(mdp3)
    for x, y, z in zip(a, b, c):
        for i in range(3):
            assert torch.equal(x[i], y[i]) and torch.equal(x[i], z[i])
    for k in sa:
        assert torch.equal(sa[k], sb[k]) and torch.equal(sa[k], sc3[k]), k
    other = make_mdp(20 if S != 20 else 12, N, 51)
    with pytest.raises(ValueError, match="checkpoint was taken with num_steps"):
        other.load_state_dict(ckpt)


# ---------------------------------------------------------------------------------------------- S = 20 control
FAST = re.compile(r"k_step<\d+, \d+, (true|false), true")  # k_step<MODE, EXACT, FULL, FAST, PACKED, PRE>
CONTROL_N = (1 << 17) + 37  # k_prepare* route, ragged last tile


def zero_length_mdp(N, seed):
    """A handle created from an AsParams whose num_steps is 0, as a caller that zero-initialises the struct makes it."""
    from allsteps_isaaclab_b200 import mdp as mdp_mod

    real = mdp_mod.make_params

    def zero_params(*a, **kw):
        p = real(*a, **kw)
        p.num_steps = 0
        return p

    mdp_mod.make_params = zero_params
    try:
        return make_mdp(20, N, seed)
    finally:
        mdp_mod.make_params = real


def control_steps(m, S, seed=61, record=None):
    """Four steps of `m`: fused, and every other one the 3-call path (device-side list) behind it.  record(fn) runs a
    step and may observe it (the kernel-name probe); returns the outputs and the final state."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    N = m.num_envs
    sc = Scenario(N, seed=seed, cfg=cfg_of(S))
    origins = sc.env_origins.cuda()
    m.generate_stones(origins)
    st = m.export_state()
    out = StepBuffers(N, "cuda:0")
    res = []
    for k in range(4):
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        views, keep = to_views(phys, origins, sc.body_indices)

        def step():
            m.step(views, keep["actions"], out)
            if k % 2:
                m.pass1(views, keep["actions"], out)
                m.reset(origins, None, out)
                m.pass2(views, out)

        (record or (lambda f: f()))(step)
        res.append(tuple(x.clone() for x in (out.obs, out.reward, out.dones)))
        st = m.export_state()
    return res, st


def test_default_length_is_the_zero_initialised_handle():
    """num_steps = 20 and num_steps = 0: the same outputs and state bit for bit."""
    mdp0 = zero_length_mdp(CONTROL_N, 61)
    assert mdp0.params.num_steps == 0 and mdp0.num_steps == 20
    ra, sa = control_steps(make_mdp(20, CONTROL_N, 61), 20)
    rb, sb = control_steps(mdp0, 20)
    for x, y in zip(ra, rb):
        assert all(torch.equal(p, q) for p, q in zip(x, y))
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k


def kernel_names_by_handle():
    """{"20" | "0" | "12" | "32": [kernel names of each control step]} from torch.profiler (run in a process of its
    own: see test_fast_instantiations_only_at_the_default_length)."""
    from torch.profiler import ProfilerActivity, profile

    def names_of(m, S):
        got = []

        def record(fn):
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            got.append([e.name for e in prof.events() if e.device_type.name == "CUDA" and "as::k_" in e.name])

        control_steps(m, S, record=record)
        return got

    return {"20": names_of(make_mdp(20, CONTROL_N, 61), 20), "0": names_of(zero_length_mdp(CONTROL_N, 61), 20),
            "12": names_of(make_mdp(12, CONTROL_N, 61), 12), "32": names_of(make_mdp(32, CONTROL_N, 61), 32)}


def test_fast_instantiations_only_at_the_default_length():
    """torch.profiler: the handles with num_steps = 20 and = 0 launch the same kernels, the FAST step-kernel
    instantiations among them; at 12 and 32 stones no FAST instantiation runs.  The profiler runs in a child process,
    so that its CUDA activity tracing does not outlive this test in the suite's process."""
    import json
    import os
    import subprocess
    import sys

    here = os.path.dirname(os.path.abspath(__file__))
    path = os.pathsep.join(p for p in (os.path.dirname(here), here, os.environ.get("PYTHONPATH")) if p)
    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--kernel-names"], capture_output=True, text=True,
                         timeout=600, env=dict(os.environ, PYTHONPATH=path))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    names = json.loads(res.stdout.strip().splitlines()[-1])
    assert names["20"] == names["0"]
    assert any(FAST.search(n) for ns in names["20"] for n in ns), f"no FAST instantiation at S = 20: {names['20']}"
    for S in ("12", "32"):
        steps = [n for ns in names[S] for n in ns if "k_step" in n]
        assert steps and not any(FAST.search(n) for n in steps), steps


# ---------------------------------------------------------------------------------------------- memory safety
@pytest.mark.parametrize("S", (3, 7, 32))
def test_guard_bands_around_workspace_and_contact_matrices(S):
    """A workspace of exactly as_workspace_bytes_for bytes and (N,1,S,3) contact matrices between guard bands: the
    fused step, the 3-call path, regeneration, export, snapshot write nothing outside them."""
    import ctypes as C

    from allsteps_isaaclab_b200 import _cabi
    from allsteps_isaaclab_b200 import mdp as mdp_mod

    for N in (300, (1 << 16) + 40):
        sc = Scenario(N, seed=71, fall_fraction=0.1, cfg=cfg_of(S))
        mdp = make_mdp(S, N, 71, intended_regen=True)
        nbytes = mdp.lib.as_workspace_bytes_for(C.byref(mdp.params), N)
        ws = Guarded((nbytes,), torch.uint8)
        mdp.lib.as_destroy(mdp.handle)
        handle = C.c_void_p()
        _cabi.check(mdp.lib.as_create(C.byref(mdp.params), N, 0, 0, ws.t.data_ptr(), nbytes, mdp._stream(),
                                      C.byref(handle)), "as_create")
        mdp.handle, mdp.workspace = handle, ws.t
        origins = sc.env_origins.cuda()
        mdp.generate_stones(origins)
        st0 = high_start(sc, S)
        mdp.import_state({k: st0[k] for k in STATE_KEYS})
        guards = [ws]
        out, gout = guarded_buffers(N, mdp_mod)
        guards += list(gout.values())
        for step in range(4):
            st = mdp.export_state()
            phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
            d = {k: v.cuda() for k, v in phys.items()}
            for k in ("force_matrix_right", "force_matrix_left"):
                g = Guarded((N, 1, S, 3), torch.float32)
                g.t.copy_(d[k])
                d[k] = g.t
                guards.append(g)
            views = mdp_mod.PhysicsViews.from_dict(d, origins, sc.body_indices)
            if step % 2 == 0:
                mdp.step(views, d["actions"], out)
            else:
                mdp.pass1(views, d["actions"], out)
                mdp.reset(origins, None, out)
                mdp.pass2(views, out)
        mdp.export_stone_poses()
        mdp.restore(mdp.snapshot())
        torch.cuda.synchronize()
        assert all(g.intact() for g in guards), f"S={S} N={N}: a guard band was written"
        assert mdp.read_stats()["step_counter"] > 0


# ---------------------------------------------------------------------------------------------- faces and misuse
def test_standalone_env_at_12_stones():
    """`StandaloneAllstepsEnv(task_cfg=AllstepsCfg(num_steps=12))`: reset() and steps through the hooks against the
    oracle, the stones written as (k,12,7) poses."""
    from allsteps_isaaclab_b200.env import StandaloneAllstepsEnv

    S, N, seed = 12, 600, 33
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.05, cfg=cfg_of(S))
    orc = ThreeCallOracle(sc, intended_regen=True)
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    robot, left, right = _fake_world(sc, phys)
    scene = types.SimpleNamespace(env_origins=sc.env_origins.cuda())
    env = StandaloneAllstepsEnv(robot, left, right, scene, "cuda:0", sc.cfg, seed=seed, intended_regen=True)
    assert env.num_steps == S
    close(env.steps_pos, orc.steps_pos, "stones of the fresh env")
    env.steps = _FakeSteps()
    o_obs = orc.reset_outside_step(phys)
    _install(robot, left, right, phys)
    obs, _ = env.reset()
    torch.cuda.synchronize()
    close_obs(obs["policy"], o_obs, "obs of the reset")
    pose, ids = env.steps.calls[0]
    assert tuple(pose.shape) == (N, S, 7)
    exact(pose[..., :3], env.steps_pos, "stone write of the reset")
    st = high_start(sc, S)
    install_mdp_state(orc, st, num_steps=S)
    env.mdp.import_state({k: st[k] for k in STATE_KEYS if k != "episode_length_buf"})
    env.episode_length_buf[:] = st["episode_length_buf"].cuda()
    busy = 0
    for step in range(8):
        env.steps.calls.clear()
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"])
        _install(robot, left, right, phys)
        obs, rew, term, to, _ = env.post_physics_step(phys["actions"].cuda())
        torch.cuda.synchronize()
        exact(term, o_term, f"step {step} terminated")
        exact(to, o_to, f"step {step} time_out")
        close(rew, o_rew, f"step {step} reward")
        close_obs(obs["policy"], o_obs, f"step {step} obs")
        exact(env.curr_target_index, orc.curr_target_index, f"step {step} curr_target_index")
        exact(env.next_target_index, orc.next_target_index, f"step {step} next_target_index")
        close(env.steps_pos, orc.steps_pos, f"step {step} stones")
        if len(o_ids):
            busy += 1
            pose, ids = env.steps.calls[0]
            assert tuple(pose.shape) == (len(o_ids), S, 7)
            exact(ids.cpu(), o_ids, f"step {step} stone write ids")
            exact(pose[..., :3], env.steps_pos[o_ids.cuda()], f"step {step} stone write")
        env.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    assert busy > 0


def test_manager_terms_at_12_stones():
    from allsteps_isaaclab_b200 import terms

    S, N, seed = 12, 700, 23
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.05, cfg=cfg_of(S))
    st0 = high_start(sc, S)
    orc = ThreeCallOracle(sc, grid_bins=7)
    install_mdp_state(orc, st0, num_steps=S)
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    robot, left, right = _fake_world(sc, phys)
    stones = _FakeSteps()
    scene = _Scene(robot=robot, foot_contacts_left=left, foot_contacts_right=right, steps=stones)
    scene.env_origins = sc.env_origins.cuda()
    env = types.SimpleNamespace(num_envs=N, device="cuda:0", scene=scene, common_step_counter=0,
                                episode_length_buf=st0["episode_length_buf"].cuda().clone(),
                                actions=torch.zeros(N, 21, device="cuda"), step_dt=4.0 / 240.0)
    b = terms.binding(env, seed=seed, task_cfg=sc.cfg, grid_bins=7)
    assert b.mdp.num_steps == S
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
            pose, got = stones.calls[0]
            assert tuple(pose.shape) == (len(ids), S, 7)
            exact(got.cpu(), ids.cpu(), f"step {step} stone write ids")
        obs = torch.cat([t(env) for t in terms.OBSERVATION_TERMS], dim=-1)
        torch.cuda.synchronize()
        close_obs(obs, o_obs, f"step {step} obs")
        exact(b.mdp.grid_state()[0], _grid_of(orc.grid)[0], f"step {step} bins")
        b.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    assert busy > 0


def test_misuse_is_refused():
    import ctypes as C

    from allsteps_isaaclab_b200 import _cabi
    from allsteps_isaaclab_b200.mdp import PhysicsViews, StepBuffers
    from allsteps_isaaclab_b200.params import make_params

    lib = _cabi.load()
    N = 256
    p = make_params(cfg_of(12))
    ws = torch.empty(lib.as_workspace_bytes_for(C.byref(p), N) + (1 << 20), dtype=torch.uint8, device="cuda")
    h = C.c_void_p()
    for bad in (2, 33):
        p.num_steps = bad
        assert lib.as_create(C.byref(p), N, 0, 0, ws.data_ptr(), ws.numel(), None, C.byref(h)) == -1
        assert b"num_steps" in lib.as_last_error()
    p.num_steps = 32
    small = lib.as_workspace_bytes(N)  # sized for 20 stones
    assert lib.as_create(C.byref(p), N, 0, 0, ws.data_ptr(), small, None, C.byref(h)) == -1
    with pytest.raises(ValueError, match="num_steps"):
        make_mdp(33, N, 1)
    mdp = make_mdp(12, N, 1)
    sc20 = Scenario(N, seed=1)
    origins = sc20.env_origins.cuda()
    mdp.generate_stones(origins)
    phys = {k: v.cuda() for k, v in sc20.physics(torch.zeros(N, 20, 3), torch.ones(N, dtype=torch.int64),
                                                  torch.zeros(N, dtype=torch.int64)).items()}
    views = PhysicsViews.from_dict(phys, origins)
    assert views.num_steps == 20
    out = StepBuffers(N, "cuda:0")
    for call in (lambda: mdp.step(views, phys["actions"], out), lambda: mdp.pass1(views, phys["actions"], out),
                 lambda: mdp.pass2(views, out)):
        with pytest.raises(ValueError, match="num_steps=12"):
            call()
    bad = dict(phys)
    bad["force_matrix_left"] = torch.zeros(N, 1, 12, 3, device="cuda")
    with pytest.raises(ValueError, match="same S"):
        PhysicsViews.from_dict(bad, origins)
    bad["force_matrix_right"] = bad["force_matrix_left"] = torch.zeros(N, 1, 33, 3, device="cuda")
    with pytest.raises(ValueError):
        PhysicsViews.from_dict(bad, origins)


if __name__ == "__main__" and "--kernel-names" in __import__("sys").argv:
    import json

    print(json.dumps(kernel_names_by_handle()))
