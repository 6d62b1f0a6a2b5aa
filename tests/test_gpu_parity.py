"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on identical replayed state.

Bar (BASELINE.json north_star): integer / index / mask outputs bit-exact; fp32 observations and rewards within
1e-5 relative (|a-b| <= 1e-5 * max(1, |b|)).
"""
from __future__ import annotations

import math

import numpy as np
import pytest
import torch

from scenario import Scenario, install_mdp_state

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def close(a: torch.Tensor, b: torch.Tensor, what: str, rtol: float = RTOL):
    a = a.detach().cpu().double()
    b = b.detach().cpu().double()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    err = (a - b).abs() / b.abs().clamp(min=1.0)
    worst = err.max().item() if err.numel() else 0.0
    assert worst <= rtol, f"{what}: max relative error {worst:.3e} > {rtol:.1e} at {int(err.argmax())}"
    return worst


def close_obs(a: torch.Tensor, b: torch.Tensor, what: str):
    """Observation compare; columns 1,2 are angles wrapped to [0, 2*pi): compare them on the circle."""
    a = a.detach().cpu().double().clone()
    b = b.detach().cpu().double().clone()
    for c in (1, 2):
        d = (a[:, c] - b[:, c]).abs()
        wrapped = torch.minimum(d, 2 * math.pi - d)
        a[:, c] = b[:, c] + wrapped
    return close(a, b, what)


def exact(a: torch.Tensor, b: torch.Tensor, what: str):
    a = a.detach().cpu()
    b = b.detach().cpu()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    bad = (a != b).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} mismatches, first at {bad[0].tolist()}"


def make_cuda(num_envs, seed, **kw):
    from allsteps_isaaclab_b200.mdp import AllstepsMDP

    return AllstepsMDP(num_envs, device="cuda:0", seed=seed, **kw)


def to_views(phys, env_origins_cuda, body_rows, layout="contiguous"):
    """Move one synthetic physics dict to the GPU in a chosen memory layout."""
    from allsteps_isaaclab_b200.mdp import PhysicsViews

    d = {k: v.cuda() for k, v in phys.items()}
    if layout == "isaac":
        # what Isaac Lab really hands out: slices of root_state_w (N,13) and body_state_w (N,B,13)
        N = d["root_pos_w"].shape[0]
        root_state = torch.zeros(N, 13, device="cuda")
        root_state[:, 0:3] = d["root_pos_w"]
        root_state[:, 3:7] = d["root_quat_w"]
        root_state[:, 7:10] = d["root_lin_vel_w"]
        root_state[:, 10:13] = d["root_ang_vel_w"]
        B = d["body_pos_w"].shape[1]
        body_state = torch.zeros(N, B, 13, device="cuda")
        body_state[..., 0:3] = d["body_pos_w"]
        d["root_pos_w"], d["root_quat_w"], d["root_lin_vel_w"] = root_state[:, 0:3], root_state[:, 3:7], root_state[:, 7:10]
        d["body_pos_w"] = body_state[..., 0:3]
        d["_keep"] = (root_state, body_state)
    elif layout == "unaligned_contact":
        # contact matrices that start 4 bytes into their allocation: the 128-bit gather path must not be taken
        keep = []
        for k in ("force_matrix_right", "force_matrix_left"):
            flat = torch.zeros(d[k].numel() + 1, device="cuda")
            flat[1:] = d[k].reshape(-1)
            d[k] = flat[1:].view(d[k].shape)
            keep.append(flat)
        d["_keep"] = tuple(keep)
    elif layout == "pinned_contact":
        for k in ("force_matrix_right", "force_matrix_left"):
            d[k] = phys[k].pin_memory()
    return PhysicsViews.from_dict(d, env_origins_cuda, body_rows), d


def compare_state(mdp, orc, what):
    st = mdp.export_state()
    exact(st["curr_target_index"], orc.curr_target_index, f"{what} curr_target_index")
    exact(st["prev_target_index"], orc.prev_target_index, f"{what} prev_target_index")
    exact(st["next_target_index"], orc.next_target_index, f"{what} next_target_index")
    exact(st["swing_leg"], orc.swing_leg, f"{what} swing_leg")
    exact(st["target_reach_count"], orc.target_reach_count, f"{what} target_reach_count")
    exact(st["episode_length_buf"], orc.episode_length_buf, f"{what} episode_length_buf")
    exact(st["curriculum"], orc.curriculum, f"{what} curriculum")
    close(st["potentials"], orc.potentials, f"{what} potentials")
    return st


def run_replay(num_envs, steps, seed, full_bodies=False, layout="contiguous", fall_fraction=0.02,
               high_index=False, per_env_levels=False, intended_regen=False, env_id_offset=0, missed_step=None):
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao

    cfg = None
    if missed_step is not None:  # extension: missed-step termination at the given foot height
        from allsteps_isaaclab_b200.config import AllstepsCfg

        cfg = AllstepsCfg(missed_step_height=missed_step)
    sc = Scenario(num_envs, seed=seed, full_bodies=full_bodies, fall_fraction=fall_fraction,
                  env_id_offset=env_id_offset, cfg=cfg)
    st0 = sc.initial_mdp_state(per_env_levels=per_env_levels)
    if high_index:
        st0["curr_target_index"] = torch.randint(11, 20, (num_envs,), generator=sc.gen)
    orc = ao.AllstepsOracle(sc.cfg, num_envs, sc.env_origins, sc.joint_limits, sc.body_indices,
                            sc.stone_uniforms(0), intended_regen=intended_regen, missed_step_height=missed_step)
    mdp = make_cuda(num_envs, seed, intended_regen=intended_regen, env_id_offset=env_id_offset, cfg=cfg,
                    missed_step=missed_step is not None)
    totals_missed = 0
    origins = sc.env_origins.cuda()
    if per_env_levels:
        # levels first, then stones at those levels (oracle: set curriculum, regenerate)
        orc.curriculum[:] = st0["curriculum"]
        orc.regenerate_stones(torch.arange(num_envs), sc.stone_uniforms(0))
        mdp.import_state({"curriculum": st0["curriculum"]})
    mdp.generate_stones(origins)  # in-kernel Philox at step counter 0
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    st = compare_state(mdp, orc, "initial")
    close(st["steps_pos"], orc.steps_pos, "initial steps_pos")
    close(st["steps_dphi"], orc.steps_dphi, "initial steps_dphi")
    # from here on both sides use the SAME stones, so that fp noise in sin/cos cannot flip a later mask
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})

    out = StepBuffers(num_envs, "cuda:0", reward_terms=True)
    totals = dict(resets=0, advanced=0, promoted=0, fixups=0, regen=0)
    worst_obs = worst_rew = 0.0
    for step in range(steps):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        mirror_u, noise_u = sc.reset_uniforms(step)
        level_before = orc.curriculum.clone()
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], mirror_u, noise_u,
                                                     sc.stone_uniforms(step))
        views, keep = to_views(phys, origins, sc.body_indices, layout)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        worst_rew = max(worst_rew, close(out.reward, o_rew, f"step {step} reward"))
        worst_obs = max(worst_obs, close_obs(out.obs, o_obs, f"step {step} obs"))
        rt = out.reward_terms.cpu()
        total = rt[:, 0] + rt[:, 1] - rt[:, 2:8].sum(-1) + rt[:, 8] + rt[:, 9]
        alive = ~o_term
        close(total[alive], o_rew[alive], f"step {step} reward terms", rtol=1e-4)
        st = compare_state(mdp, orc, f"step {step}")
        # reset rows
        n_reset = int(out.n_reset.item())
        assert n_reset == len(o_ids), f"step {step}: n_reset {n_reset} vs {len(o_ids)}"
        ids = out.reset_ids[:n_reset].long().sort().values
        exact(ids, o_ids, f"step {step} reset ids")
        if n_reset:
            w = orc.reset_writes
            root = torch.cat((w["root_pose"], w["root_velocity"]), dim=-1)
            close(out.reset_root_state[ids], root, f"step {step} reset root_state")
            close(out.reset_joint_pos[ids], w["joint_pos"], f"step {step} reset joint_pos")
            close(out.reset_joint_vel[ids], w["joint_vel"], f"step {step} reset joint_vel")
        if intended_regen and n_reset and len(orc.regenerated_ids):
            close(st["steps_pos"], orc.steps_pos, f"step {step} regenerated steps_pos")
            close(st["steps_dphi"], orc.steps_dphi, f"step {step} regenerated steps_dphi")
            mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
            totals["regen"] += len(orc.regenerated_ids)
        stats = mdp.read_stats()
        assert stats["n_reset"] == len(o_ids)
        assert stats["n_terminated"] == int(o_term.sum())
        assert stats["n_time_out"] == int(o_to.sum())
        assert stats["sum_target_index"] == int(orc.pass1["curr_target_index"].sum())
        if missed_step is not None:
            assert stats["n_missed"] == int(orc.missed_step_pass1.sum()), f"step {step} n_missed"
            totals["missed"] = totals.get("missed", 0) + stats["n_missed"]
        else:
            assert stats["n_missed"] == 0
        totals["resets"] += n_reset
        totals["advanced"] += stats["n_advanced"]
        totals["promoted"] += int((orc.curriculum != level_before).any())
        totals["fixups"] += int(n_reset == 0)
    return totals, worst_obs, worst_rew


@pytest.mark.parametrize("layout", ["contiguous", "unaligned_contact", "pinned_contact", "isaac"])
def test_separate_contact_gather_kernels(layout):
    """From 2^17 envs on the current stone's contact vectors are gathered by a kernel of their own: two lanes per env
    on 16-byte aligned rows (device or pinned host memory), one lane per env otherwise.  "isaac": slices of one (N,13)
    root_state_w and of the full (N,17,13) body_state_w -- the root rows travel as one bulk copy (packed tile), the
    three body rows are gathered by k_body_gather into a dense array first."""
    totals, _, _ = run_replay((1 << 17) + 37, 2, seed=29, layout=layout, high_index=(layout == "contiguous"),
                              full_bodies=(layout == "isaac"))
    assert totals["advanced"] > 0


@pytest.mark.parametrize("num_envs,steps", [(64, 40), (4096, 12)])
def test_fused_step_matches_oracle(num_envs, steps):
    totals, wo, wr = run_replay(num_envs, steps, seed=11)
    assert totals["resets"] > 0 and totals["advanced"] > 0
    print(f"N={num_envs}: {totals}, worst obs rel err {wo:.2e}, reward {wr:.2e}")


def test_ragged_tile_and_isaac_strided_views():
    # 1001 envs: last CTA has 105 valid rows (not a multiple of 4) -> cooperative path; (N,13) strided root views,
    # full 17-body tensor with 13-float rows -> strided gathers
    totals, _, _ = run_replay(1001, 10, seed=5, full_bodies=True, layout="isaac")
    assert totals["resets"] > 0


def test_full_body_tensor_contiguous():
    totals, _, _ = run_replay(640, 8, seed=6, full_bodies=True)
    assert totals["resets"] > 0


def test_no_reset_steps_skip_pass2():
    # nothing falls and episodes are young in most steps at N=64 => the reference runs a single pass (DRL:360);
    # the CUDA path must take its fix-up route and still match bit for bit
    totals, _, _ = run_replay(64, 30, seed=3, fall_fraction=0.0)
    assert totals["fixups"] > 0


def test_curriculum_promotion_rule():
    totals, _, _ = run_replay(512, 14, seed=8, high_index=True)
    assert totals["promoted"] > 0


def test_per_env_levels_and_env_id_offset():
    totals, _, _ = run_replay(384, 8, seed=21, per_env_levels=True, env_id_offset=1 << 20)
    assert totals["resets"] > 0


@pytest.mark.parametrize("regen_mode", ["1", "2"])
def test_intended_regeneration_extension(regen_mode, monkeypatch):
    # k_reset_rows regenerates with one warp per env (short lists) or one thread per env (long lists): both shapes
    monkeypatch.setenv("ALLSTEPS_REGEN_MODE", regen_mode)
    totals, _, _ = run_replay(768, 10, seed=9, high_index=True, intended_regen=True, per_env_levels=True)
    assert totals["regen"] > 0


def test_long_replay_over_whole_episodes():
    """A soak: 1200 consecutive steps of 192 envs against the oracle, state compared after every step -- longer than an
    episode (900 steps), so every env times out or falls and restarts several times, the episode counters run their
    whole range and the promotion rule is evaluated on every reset."""
    totals, _, _ = run_replay(192, 1200, seed=123, fall_fraction=0.004)
    assert totals["resets"] > 400 and totals["advanced"] > 10000


def test_missed_step_termination_extension():
    """BASELINE north_star "missed-step termination" (no reference counterpart, SURVEY D4): AS_FLAG_MISSED_STEP against
    the oracle's specification of it -- masks bit-exact; off by default (every other replay asserts n_missed == 0)."""
    # the synthetic swing foot hovers 0.11 m above its stone: 0.12 makes every foot outside the radius a missed step
    totals, _, _ = run_replay(2048, 8, seed=61, missed_step=0.12)
    assert totals["missed"] > 1000 and totals["resets"] >= totals["missed"]
    # at the default height nothing of the synthetic state counts as down: the flag alone changes nothing
    totals, _, _ = run_replay(1024, 4, seed=62, missed_step=0.05)
    assert totals["missed"] == 0 and totals["resets"] > 0


def test_explicit_stone_uniforms():
    from oracle import allsteps_oracle as ao

    sc = Scenario(300, seed=2)
    levels = torch.randint(0, 10, (300,), generator=sc.gen)
    u = torch.rand(5, 300, 20, generator=sc.gen)
    pos, dphi = ao.generate_stones(sc.cfg, levels, u)
    pos = pos + sc.env_origins[:, None, :]
    mdp = make_cuda(300, 2)
    mdp.import_state({"curriculum": levels})
    mdp.generate_stones(sc.env_origins.cuda(), uniforms=u.cuda())
    st = mdp.export_state()
    close(st["steps_pos"], pos, "steps_pos")
    close(st["steps_dphi"], dphi, "steps_dphi")
    # a subset regenerated with other draws leaves the rest untouched
    ids = torch.tensor([3, 17, 299])
    u2 = torch.rand(5, 300, 20, generator=sc.gen)
    pos2, _ = ao.generate_stones(sc.cfg, levels, u2)
    pos2 = pos2 + sc.env_origins[:, None, :]
    mdp.generate_stones(sc.env_origins.cuda(), env_ids=ids.cuda(), uniforms=u2.cuda())
    st2 = mdp.export_state()
    expect = pos.clone()
    expect[ids] = pos2[ids]
    close(st2["steps_pos"], expect, "steps_pos after partial regeneration")


@pytest.mark.parametrize("N,fall,layout,steps", [(1536, 0.02, "contiguous", 8), (48, 0.0, "contiguous", 12),
                                                 (160, 0.004, "contiguous", 1000),  # a soak: longer than an episode
                                                 ((1 << 17) + 37, 0.02, "contiguous", 4),
                                                 (1 << 17, 0.02, "isaac", 3)])
def test_three_call_path_matches_oracle(N, fall, layout, steps):
    """pass1 / reset / pass2 with the caller doing the 'PhysX writes' in between (the DirectRLEnv hook order).  Pass 1
    speculates pass 2 for the envs that do not reset; pass2 redoes the ones that did from the written-back state,
    no_reset takes the speculation back (the 48-env quiet case: most steps have no reset).  From 2^17 envs on the
    prepared instantiations run (k_prepare* + the step kernel without scattered accesses)."""
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao

    seed = 13
    sc = Scenario(N, seed=seed, fall_fraction=fall, full_bodies=(layout == "isaac"))
    st0 = sc.initial_mdp_state()
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    mdp = make_cuda(N, seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    ep_len = st0["episode_length_buf"].cuda()
    n_quiet = n_busy = 0
    for step in range(steps):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        # pass1 advances the step counter, so the reset that follows draws at step + 1
        mirror_u, noise_u = sc.reset_uniforms(step + 1)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], mirror_u, noise_u, None)
        views, keep = to_views(phys, origins, sc.body_indices, layout)
        n_quiet += int(len(o_ids) == 0)
        n_busy += int(len(o_ids) > 0)
        ep_len += 1  # DRL:351
        mdp.pass1(views, keep["actions"], out, episode_length=ep_len)
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        close(out.reward, o_rew, f"step {step} reward")
        ids = (out.terminated | out.time_out).nonzero().squeeze(-1)  # DRL:359
        exact(ids, o_ids, f"step {step} ids")
        if len(ids):
            mdp.reset(origins, ids, out, episode_length=ep_len)
            k = len(ids)
            w = orc.reset_writes
            close(out.reset_root_state[:k], torch.cat((w["root_pose"], w["root_velocity"]), -1), "root rows")
            close(out.reset_joint_pos[:k], w["joint_pos"], "joint_pos rows")
            # the PhysX writes (ART:316-489): data views change for the reset rows; contacts are zeroed
            keep["root_pos_w"][ids] = out.reset_root_state[:k, 0:3]
            keep["root_quat_w"][ids] = out.reset_root_state[:k, 3:7]
            keep["root_lin_vel_w"][ids] = out.reset_root_state[:k, 7:10]
            keep["joint_pos"][ids] = out.reset_joint_pos[:k]
            keep["joint_vel"][ids] = out.reset_joint_vel[:k]
            keep["force_matrix_right"][ids] = 0.0
            keep["force_matrix_left"][ids] = 0.0
            mdp.pass2(views, out)
        else:
            mdp.no_reset()  # DRL:360: `_reset_idx` is skipped, the observations of pass 1 stand
        torch.cuda.synchronize()
        close_obs(out.obs, o_obs, f"step {step} obs")
        exact(ep_len, orc.episode_length_buf, f"step {step} episode_length")
        st = mdp.export_state()
        exact(st["curr_target_index"], orc.curr_target_index, f"step {step} idx")
        exact(st["swing_leg"], orc.swing_leg, f"step {step} leg")
        exact(st["target_reach_count"], orc.target_reach_count, f"step {step} count")
        exact(st["curriculum"], orc.curriculum, f"step {step} curriculum")
        close(st["potentials"], orc.potentials, f"step {step} potentials")
    assert n_busy > 0 or fall == 0.0
    if fall == 0.0:
        assert n_quiet > 0, "the quiet case is there to exercise as_step_no_reset"


def test_export_state_of_selected_fields():
    """`export_state(fields)` materialises only what is asked for (the env properties of the hooks use it), with the
    same values as the full export."""
    mdp = make_cuda(500, 5)
    mdp.generate_stones(torch.zeros(500, 3, device="cuda"))
    full = mdp.export_state()
    one = mdp.export_state(("potentials",))
    assert set(one) == {"potentials"} and torch.equal(one["potentials"], full["potentials"])
    some = mdp.export_state(("next_target_index", "steps_dphi"))
    assert set(some) == {"curr_target_index", "prev_target_index", "next_target_index", "steps_dphi"}
    for k, v in some.items():
        assert torch.equal(v, full[k]), k
    with pytest.raises(KeyError):
        mdp.export_state(("no_such_buffer",))


def test_action_path_and_mirror_rows():
    from oracle import allsteps_oracle as ao

    N = 777
    sc = Scenario(N, seed=4)
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, None)
    levels = torch.randint(0, 10, (N,), generator=sc.gen)
    orc.curriculum[:] = levels
    actions = -1.5 + 3.0 * torch.rand(N, 21, generator=sc.gen)
    orc.clamp_actions(actions)
    mdp = make_cuda(N, 4)
    mdp.import_state({"curriculum": levels})
    eff = mdp.apply_action(actions.cuda())  # 777 envs: six 128-env tiles by TMA bulk copies + 9 envs element by element
    close(eff, orc.joint_efforts(), "joint efforts")
    # a strided (N,32) view and a view 4 bytes into an allocation take the element loop: same bits
    wide = torch.zeros(N, 32, device="cuda")
    wide[:, :21] = actions.cuda()
    exact(mdp.apply_action(wide[:, :21]), eff, "efforts from a strided action view")
    pad = torch.empty(N * 21 + 1, device="cuda")
    off = pad[1:].view(N, 21)
    off.copy_(actions)
    exact(mdp.apply_action(off), eff, "efforts from a misaligned action view")
    # mirror augmentation, ENV:570-660: against the oracle's restatement (pinned to the live reference functions in
    # tests/test_oracle_vs_reference.py and to tests/golden/mirror_symmetry.npz)
    cfg = sc.cfg
    tabs = (cfg.right_joint_indices, cfg.left_joint_indices, cfg.negation_joint_indices)
    obs = torch.randn(N, 59, generator=sc.gen)
    exact(mdp.mirror_rows(obs.cuda(), "obs"), ao.symmetric_states(obs, *tabs, "obs"), "mirrored observations")
    exact(mdp.mirror_rows(actions.cuda(), "actions"), ao.symmetric_states(actions, *tabs, "actions"),
          "mirrored actions")


@pytest.mark.parametrize("rows", [4 * 128, 3 * 128 + 44, 1029, 127, 32 * 4096])
def test_mirror_kernel_tiles_and_tails(rows):
    """k_mirror_batch moves full 128-row tiles through shared memory (TMA bulk copies) and the rest element by element:
    whole tiles, tiles + a tail, a row count that puts the lower half off a 16-byte boundary (element loop for
    everything), fewer rows than a tile, a rollout-sized batch; and inputs that are not 16-byte aligned.  Against the
    oracle's restatement of ENV:570-660 (pinned to the live reference), bit for bit incl. NaN / -0.0 / inf entries."""
    from allsteps_isaaclab_b200 import symmetry
    from oracle import allsteps_oracle as ao

    mdp = make_cuda(64, 3)
    cfg = mdp.cfg
    tabs = (cfg.right_joint_indices, cfg.left_joint_indices, cfg.negation_joint_indices)
    g = torch.Generator().manual_seed(rows)
    obs = torch.randn(rows, 59, generator=g)
    act = torch.randn(rows, 21, generator=g)
    mus = torch.randn(rows, 21, generator=g)
    for t in (obs, act, mus):
        flat = t.view(-1)
        flat[::97] = float("nan")
        flat[5::101] = -0.0
        flat[7::103] = float("inf")
    bits = lambda t: t.detach().cpu().contiguous().numpy().view(np.uint32)  # noqa: E731
    want = (ao.symmetric_states(obs, *tabs, "obs"), ao.symmetric_states(act, *tabs, "actions"),
            ao.symmetric_states(mus, *tabs, "actions"))
    l0 = mdp.launch_count
    got = symmetry.mirror_batch(mdp, obs.cuda(), act.cuda(), mus.cuda())
    assert mdp.launch_count == l0 + 1
    for w, o in zip(want, got):
        assert np.array_equal(bits(o), bits(w))
    assert np.array_equal(bits(mdp.mirror_rows(obs.cuda(), "obs")), bits(want[0]))
    # a view that starts 4 bytes into an allocation: no bulk copies possible, same result
    pad = torch.empty(rows * 59 + 1, device="cuda")
    view = pad[1:].view(rows, 59)
    view.copy_(obs)
    assert np.array_equal(bits(mdp.mirror_rows(view, "obs")), bits(want[0]))


def test_symmetry_functions_match_the_reference_fixture():
    """SURVEY 8 f1: the drop-ins with the reference's signatures (ENV:570, ENV:611) and the play_steps-shaped call
    (learning/a2c_ppo_mirroring.py:20-40) against outputs of the reference's own functions (mirror_symmetry.npz),
    bit for bit (-0.0, inf and NaN entries included)."""
    import types

    import numpy as np

    import golden_util as gu
    from allsteps_isaaclab_b200 import symmetry
    from allsteps_isaaclab_b200.config import AllstepsCfg

    d = gu.load("mirror_symmetry.npz")
    bits = lambda t: t.detach().cpu().contiguous().numpy().view(np.uint32)  # noqa: E731
    f = lambda k: torch.from_numpy(d[k].view(np.float32).copy()).cuda()  # noqa: E731
    cfg = AllstepsCfg()
    base = types.SimpleNamespace(
        right_body_indices=torch.tensor(cfg.right_joint_indices, device="cuda"),
        left_body_indices=torch.tensor(cfg.left_joint_indices, device="cuda"),
        negation_body_indices=torch.tensor(cfg.negation_joint_indices, device="cuda"),
        observation_space=types.SimpleNamespace(shape=(8, 59)), action_space=types.SimpleNamespace(shape=(8, 21)),
        device="cuda:0")
    env = types.SimpleNamespace(unwrapped=base, device="cuda:0")
    obs, actions, mus = f("obs"), f("actions"), f("mus")
    mdp0 = symmetry._mdp_for(env)
    l0 = mdp0.launch_count
    o, a, m = symmetry.get_symmetric_states_rl_games(obs, actions, env, False, mus)
    assert mdp0.launch_count == l0 + 1, "obses, actions and mus must be mirrored by ONE launch"
    assert np.array_equal(bits(o), d["rl_games_obs"]) and np.array_equal(bits(a), d["rl_games_actions"])
    assert np.array_equal(bits(m), d["rl_games_mus"])
    o, a = symmetry.get_symmetric_states_rsl_rl(obs, actions, env)
    assert np.array_equal(bits(o), d["rsl_rl_obs"]) and np.array_equal(bits(a), d["rsl_rl_actions"])
    o, a, m = symmetry.get_symmetric_states_rl_games(None, actions, env, False, None)
    assert o is None and m is None and np.array_equal(bits(a), d["actions_only"])
    # A2CAgentSymmetry.play_steps, learning/a2c_ppo_mirroring.py:23-38
    R = obs.shape[0]
    batch = {"returns": torch.randn(R, 1, device="cuda"), "dones": torch.zeros(R, device="cuda"),
             "values": torch.randn(R, 1, device="cuda"), "sigmas": torch.randn(R, 21, device="cuda"),
             "neglogpacs": torch.randn(R, device="cuda"), "obses": obs, "actions": actions, "mus": mus,
             "played_frames": R}
    ret0 = batch["returns"].clone()
    out = symmetry.augment_play_steps_batch(batch, env)
    assert out["returns"].shape == (2 * R, 1) and torch.equal(out["returns"][R:], ret0)
    assert out["dones"].shape == (2 * R,) and out["neglogpacs"].shape == (2 * R,) and out["sigmas"].shape == (2 * R, 21)
    assert np.array_equal(bits(out["obses"]), d["rl_games_obs"]) and np.array_equal(bits(out["mus"]), d["rl_games_mus"])
    # an env whose index tensors are not the ones the kernels are built with is refused
    fields = {k: v for k, v in base.__dict__.items() if not k.startswith("_allsteps")}
    bad = types.SimpleNamespace(unwrapped=types.SimpleNamespace(**{**fields,
                                "right_body_indices": base.left_body_indices}), device="cuda:0")
    with pytest.raises(ValueError, match="mirror tables"):
        symmetry.get_symmetric_states_rsl_rl(obs, actions, bad)
    # the hooks' env serves its own handle
    big = torch.randn(32 * 4096, 59, device="cuda")
    o2, _ = symmetry.get_symmetric_states_rsl_rl(big, None, env)
    torch.cuda.synchronize()
    exact(o2, ao_sym(big.cpu(), cfg), "32 x 4096 observation rows (one PPO epoch at rl_games' default scale)")


def ao_sym(x, cfg):
    from oracle import allsteps_oracle as ao

    return ao.symmetric_states(x, cfg.right_joint_indices, cfg.left_joint_indices, cfg.negation_joint_indices, "obs")


def test_joint_scaling_is_bit_exact():
    """The kernel divides with precomputed reciprocals + a two-FMA correction (csrc scale_joint); the quotient must
    be the correctly rounded one, i.e. bit-identical to torch's `2*(x-offset)/(hi-lo)` (feeds the at-limit count)."""
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao

    N = 1 << 18
    sc = Scenario(N, seed=77)
    mdp = make_cuda(N, 77, skip_pass2=True)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    st = mdp.export_state()
    out = StepBuffers(N, "cuda:0", reset_rows=False)
    lim = sc.joint_limits
    for rep in range(3):
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        span = lim[:, 1] - lim[:, 0]
        if rep == 1:  # hug the limits, where |scaled| ~ 0.99 .. 1.01 decides the at-limit count
            side = torch.randint(0, 2, (N, 21), generator=sc.gen).float()
            phys["joint_pos"] = lim[:, 0] + side * span + (torch.rand(N, 21, generator=sc.gen) - 0.5) * 0.02 * span
        if rep == 2:  # wide dynamic range incl. tiny values
            phys["joint_pos"] = torch.randn(N, 21, generator=sc.gen) * torch.logspace(-6, 1, 21)
        views, keep = to_views(phys, origins, sc.body_indices)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        expect = ao.scale_to_unit(phys["joint_pos"], lim[:, 0], lim[:, 1])
        keep_rows = ~(out.terminated | out.time_out).cpu()  # reset rows show the start pose instead
        got = out.obs[:, 6:27].cpu()
        assert torch.equal(got[keep_rows], expect[keep_rows]), "joint_pos_scaled is not bit-identical to torch"


def test_true_division_fallback_kernels():
    """A divisor with an all-ones significand is the excluded case of the two-FMA quotient (Markstein): as_create
    then selects the step-kernel instantiations that divide.  One joint is given such a range (upper - lower =
    0x3fffffff); full tiles, a ragged tail, resets and the bit-exact joint scaling must all still match the oracle.
    Two sizes: one that gathers inside the step kernel, and one from which k_prepare* gathers for it."""
    from allsteps_isaaclab_b200.config import AllstepsCfg
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers
    from oracle import allsteps_oracle as ao

    class Cfg(AllstepsCfg):
        def joint_limits_rad(self):
            lim = list(super().joint_limits_rad())
            lim[9] = (0.0, 1.9999998807907104)  # fp32 0x3fffffff
            return lim

    seed, cfg = 53, Cfg()
    for N in (300, (1 << 16) + 44):
        sc = Scenario(N, seed=seed, cfg=cfg, fall_fraction=0.1)
        rng = (sc.joint_limits[9, 1] - sc.joint_limits[9, 0]).view(torch.int32).item()
        assert rng & 0x7FFFFF == 0x7FFFFF, "the test's joint range is not the excluded case"
        st0 = sc.initial_mdp_state()
        orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
        mdp = AllstepsMDP(N, device="cuda:0", cfg=cfg, seed=seed)
        origins = sc.env_origins.cuda()
        mdp.generate_stones(origins)
        install_mdp_state(orc, st0)
        mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                              "episode_length_buf", "potentials")})
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        out = StepBuffers(N, "cuda:0")
        resets = 0
        for step in range(4):
            phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
            mirror_u, noise_u = sc.reset_uniforms(step)
            o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], mirror_u, noise_u,
                                                         sc.stone_uniforms(step))
            views, keep = to_views(phys, origins, sc.body_indices)
            mdp.step(views, keep["actions"], out)
            torch.cuda.synchronize()
            at = f"N {N} step {step}"
            exact(out.terminated, o_term, f"{at} terminated")
            exact(out.time_out, o_to, f"{at} time_out")
            close(out.reward, o_rew, f"{at} reward")
            close_obs(out.obs, o_obs, f"{at} obs")
            compare_state(mdp, orc, at)
            keep_rows = ~(o_term | o_to)
            expect = ao.scale_to_unit(phys["joint_pos"], sc.joint_limits[:, 0], sc.joint_limits[:, 1])
            assert torch.equal(out.obs[:, 6:27].cpu()[keep_rows], expect[keep_rows]), f"{at}: joint_pos_scaled is not bit-identical"
            resets += len(o_ids)
        assert resets > 0


def test_straight_line_math_is_exact(tmp_path):
    """The kernels compute sqrt and the constant-divisor quotients as straight-line code (csrc/as_math.cuh: no range
    check, no branch to a slow path).  tools/exact_math_check.cu compares them on the device with the IEEE operations
    they replace: sqrt_rn against sqrtf for ALL 2^32 inputs, div_by_const against `/` for step_dt and the task's joint
    ranges, div_with_rcp against `/` for quaternion-like operands.  Zero mismatches required."""
    import os
    import shutil
    import subprocess

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(nvcc):
        pytest.skip("nvcc not available on this box")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "exact_math_check")
    build = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-fmad=false",
                            "-o", exe, os.path.join(root, "tools", "exact_math_check.cu")],
                           capture_output=True, text=True)
    assert build.returncode == 0, build.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout + run.stderr
    assert run.stdout.count(" 0 mismatches") == 4, run.stdout


def test_cuda_graph_replay_is_identical_to_eager_steps():
    """The launch-bound small-N regime runs the step as one captured CUDA graph; results must not change."""
    from allsteps_isaaclab_b200.mdp import PhysicsViews, StepBuffers

    N, seed = 4096, 41
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    origins = sc.env_origins.cuda()
    mdps = [make_cuda(N, seed) for _ in range(2)]
    for m in mdps:
        m.generate_stones(origins)
        m.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                            "episode_length_buf", "potentials")})
    stones = mdps[0].export_state()["steps_pos"].cpu()
    phys = sc.physics(stones, st0["curr_target_index"], st0["swing_leg"])
    static = {k: v.cuda() for k, v in phys.items()}          # the graph is bound to these tensors
    views = PhysicsViews.from_dict(static, origins, sc.body_indices)
    out_g, out_e = StepBuffers(N, "cuda:0"), StepBuffers(N, "cuda:0")
    step = mdps[0].capture_step(views, static["actions"], out_g)
    assert step.kernels_per_replay >= 2
    for i in range(6):
        st = mdps[1].export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        for k, v in phys.items():
            static[k].copy_(v)                                # "physics" writes in place
        step.replay()
        mdps[1].step(views, static["actions"], out_e)
        torch.cuda.synchronize()
        for name in ("obs", "reward", "terminated", "time_out", "reset_root_state", "reset_joint_pos"):
            g, e = getattr(out_g, name), getattr(out_e, name)
            if not torch.equal(g, e):
                bad = (g != e).nonzero()
                vals = [(g[tuple(b)].item(), e[tuple(b)].item()) for b in bad[:8]]
                raise AssertionError(f"step {i}: {name} differs at {len(bad)} places, first {bad[:8].tolist()}: {vals}; "
                                     f"n_reset graph/eager = {int(out_g.n_reset)}/{int(out_e.n_reset)}")
        a, b = mdps[0].export_state(), mdps[1].export_state()
        for k in a:
            assert torch.equal(a[k], b[k]), f"step {i}: state {k}"
        assert mdps[0].read_stats()["step_counter"] == mdps[1].read_stats()["step_counter"]


@pytest.mark.parametrize("regen_mode,N,steps", [("0", 3000, 10), ("1", 3000, 10), ("2", 3000, 10), ("0", 700, 300)])
def test_grid_curriculum_extension(regen_mode, N, steps, monkeypatch):
    """Kernel (c): difficulty histogram + inverse-CDF bin sampling + regeneration at the bin's difficulty.  No
    reference counterpart: checked bit for bit against its specification, oracle/grid_curriculum.py.  (regen_mode:
    the shape of k_reset_rows -- chosen by list length, one warp per env, one thread per env.)"""
    monkeypatch.setenv("ALLSTEPS_REGEN_MODE", regen_mode)
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao
    from oracle import grid_curriculum as gc

    seed, B = 19, 11
    sc = Scenario(N, seed=seed, fall_fraction=0.05)
    st0 = sc.initial_mdp_state()
    grid = gc.GridCurriculum(N, B)
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0),
                            grid=grid, seed=seed)
    mdp = make_cuda(N, seed, grid_bins=B)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    total_reset = 0
    for step in range(steps):  # (the 300-step case: histograms that have grown for a while, many sampled bins)
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(step))
        views, keep = to_views(phys, origins, sc.body_indices)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        close(out.reward, o_rew, f"step {step} reward")
        close_obs(out.obs, o_obs, f"step {step} obs")
        bins, att, succ = mdp.grid_state()
        exact(bins, torch.from_numpy(grid.bins.copy()), f"step {step} bins")
        exact(att, torch.from_numpy(grid.attempts.astype(np.int64)), f"step {step} attempts histogram")
        exact(succ, torch.from_numpy(grid.successes.astype(np.int64)), f"step {step} successes histogram")
        st = compare_state(mdp, orc, f"step {step}")
        close(st["steps_pos"], orc.steps_pos, f"step {step} regenerated stones")
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        total_reset += len(o_ids)
    assert total_reset > 500 and int(att.sum()) == total_reset
    assert len(np.unique(grid.bins)) > 30  # the sampler spreads over the grid


@pytest.mark.parametrize("num_envs", [1, 3, 5, 127, 129])
def test_tiny_and_ragged_env_counts(num_envs):
    # fewer envs than a tile, not a multiple of 4 (no TMA for the ragged tile), one more than a tile
    run_replay(num_envs, 6, seed=100 + num_envs, fall_fraction=0.2)


def test_reset_with_empty_id_list_is_a_no_op():
    from allsteps_isaaclab_b200.mdp import StepBuffers

    mdp = make_cuda(64, 1)
    origins = torch.zeros(64, 3, device="cuda")
    mdp.generate_stones(origins)
    before = mdp.export_state()
    n0 = mdp.launch_count
    mdp.reset(origins, torch.zeros(0, dtype=torch.long, device="cuda"), StepBuffers(64, "cuda:0"))
    assert mdp.launch_count == n0  # DRL:360: `_reset_idx` is not entered for an empty id list
    after = mdp.export_state()
    for k in before:
        assert torch.equal(before[k], after[k])


def test_api_misuse_is_reported():
    from allsteps_isaaclab_b200 import _cabi
    from allsteps_isaaclab_b200.mdp import PhysicsViews, StepBuffers

    N = 256
    sc = Scenario(N, seed=1)
    mdp = make_cuda(N, 1)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    st = mdp.export_state()
    phys = {k: v.cuda() for k, v in sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(),
                                               st["swing_leg"].cpu()).items()}
    views = PhysicsViews.from_dict(phys, origins)
    out = StepBuffers(N, "cuda:0")
    mdp.pass2(views, out)  # pass 2 without pass 1 is legal: DirectRLEnv.reset() -> _reset_idx -> ENV:567
    mdp.step(views, phys["actions"], out, finish=False)
    with pytest.raises(_cabi.AllstepsLibraryError, match="as_finish_step"):
        mdp.pass2(views, out)  # ... but not while a fused step is open
    with pytest.raises(_cabi.AllstepsLibraryError, match="as_finish_step"):
        mdp.step(views, phys["actions"], out)  # a fused step is still open
    with pytest.raises(_cabi.AllstepsLibraryError):
        mdp.export_state()
    mdp.finish_step()
    with pytest.raises(_cabi.AllstepsLibraryError):
        mdp.finish_step()  # nothing to close
    with pytest.raises(ValueError):
        mdp.step(PhysicsViews.from_dict({k: v[:128] for k, v in phys.items()}, origins[:128]), phys["actions"], out)
    with pytest.raises(TypeError):
        mdp.step(views, phys["actions"].double(), out)


def test_one_million_envs_against_the_oracle_and_invariants():
    """BASELINE.json's full size.  Two steps against the CPU oracle, plus size-independent properties: results do not
    depend on how the envs are sharded (env-id offset + Philox keyed by global id), and a rigid translation of the
    whole world leaves the root-frame observation unchanged."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers
    from oracle import allsteps_oracle as ao

    N, seed = 1 << 20, 5
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    install_mdp_state(orc, st0)
    mdp = make_cuda(N, seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    keys = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")
    mdp.import_state({k: st0[k] for k in keys})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    # the same envs as two shards of 512K with their own handles
    half = N // 2
    shards = [AllstepsMDP(half, device="cuda:0", seed=seed, env_id_offset=r * half) for r in range(2)]
    for r, sh in enumerate(shards):
        sl = slice(r * half, (r + 1) * half)
        sh.import_state({k: st0[k][sl] for k in keys})
        sh.import_state({"steps_pos": orc.steps_pos[sl], "steps_dphi": orc.steps_dphi[sl]})
    out = StepBuffers(N, "cuda:0")
    outs = [StepBuffers(half, "cuda:0") for _ in range(2)]
    for step in range(2):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, None)
        views, keep = to_views(phys, origins, sc.body_indices)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        close(out.reward, o_rew, f"step {step} reward")
        close_obs(out.obs, o_obs, f"step {step} obs")
        compare_state(mdp, orc, f"step {step}")
        assert int(out.n_reset.item()) == len(o_ids)
        for r, sh in enumerate(shards):
            sl = slice(r * half, (r + 1) * half)
            v, k = to_views({kk: vv[sl] for kk, vv in phys.items()}, origins[sl].contiguous(), sc.body_indices)
            sh.step(v, k["actions"], outs[r])
            torch.cuda.synchronize()
            for name in ("obs", "reward", "terminated", "time_out", "reset_joint_pos", "reset_root_state"):
                assert torch.equal(getattr(outs[r], name), getattr(out, name)[sl]), f"shard {r} step {step}: {name}"
    # translation invariance of the root-frame part of the observation (columns 50..58) and of everything else
    shift = torch.tensor([8.0, -16.0, 2.0])
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    a = make_cuda(4096, seed, skip_pass2=True)
    b = make_cuda(4096, seed, skip_pass2=True)
    sub = slice(0, 4096)
    st = {k: getattr(orc, k)[sub] for k in ("curr_target_index", "swing_leg", "target_reach_count", "potentials")}
    st["episode_length_buf"] = orc.episode_length_buf[sub]
    a.import_state({**st, "steps_pos": orc.steps_pos[sub], "steps_dphi": orc.steps_dphi[sub]})
    b.import_state({**st, "steps_pos": orc.steps_pos[sub] + shift, "steps_dphi": orc.steps_dphi[sub]})
    pa = {k: v[sub].clone() for k, v in phys.items()}
    pb = {k: v[sub].clone() for k, v in phys.items()}
    pb["root_pos_w"] = pb["root_pos_w"] + shift
    pb["body_pos_w"] = pb["body_pos_w"] + shift
    pb["root_pos_w"][:, 2] -= shift[2]  # keep the absolute-height termination (root z < 0.4) the same ...
    pb["body_pos_w"][:, :, 2] -= shift[2]  # ... by translating in the horizontal plane only
    stones_b = orc.steps_pos[sub].clone()
    stones_b[..., :2] += shift[:2]
    b.import_state({"steps_pos": stones_b})
    oa, ob = StepBuffers(4096, "cuda:0"), StepBuffers(4096, "cuda:0")
    va, ka = to_views(pa, origins[sub].contiguous(), sc.body_indices)
    vb, kb = to_views(pb, (sc.env_origins[sub] + torch.tensor([shift[0], shift[1], 0.0])).cuda().contiguous(),
                      sc.body_indices)
    a.step(va, ka["actions"], oa)
    b.step(vb, kb["actions"], ob)
    torch.cuda.synchronize()
    exact(oa.terminated, ob.terminated, "translated world: terminated")
    keep_rows = ~(oa.terminated | oa.time_out).cpu()
    assert torch.allclose(oa.obs.cpu()[keep_rows], ob.obs.cpu()[keep_rows], atol=2e-4, rtol=0)
    # the progress term is 60 x a difference of distances of world coordinates ~1e3 m (fp32 ulp 1e-4)
    assert torch.allclose(oa.reward.cpu()[keep_rows], ob.reward.cpu()[keep_rows], atol=5e-2, rtol=0)


def test_pinned_host_contact_matrices_are_read_in_place():
    """Zero-copy ingest: the (N,1,20,3) contact matrices stay in pinned host memory; results are unchanged."""
    from allsteps_isaaclab_b200.mdp import PhysicsViews, StepBuffers

    N, seed = 5000, 77
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    origins = sc.env_origins.cuda()
    mdps = [make_cuda(N, seed) for _ in range(2)]
    for m in mdps:
        m.generate_stones(origins)
        m.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                            "episode_length_buf", "potentials")})
    outs = [StepBuffers(N, "cuda:0"), StepBuffers(N, "cuda:0")]
    for step in range(4):
        st = mdps[0].export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        dev = {k: v.cuda() for k, v in phys.items()}
        mixed = dict(dev)
        mixed["force_matrix_right"] = phys["force_matrix_right"].pin_memory()
        mixed["force_matrix_left"] = phys["force_matrix_left"].pin_memory()
        mdps[0].step(PhysicsViews.from_dict(dev, origins), dev["actions"], outs[0])
        mdps[1].step(PhysicsViews.from_dict(mixed, origins), dev["actions"], outs[1])
        torch.cuda.synchronize()
        for name in ("obs", "reward", "terminated", "time_out"):
            assert torch.equal(getattr(outs[0], name), getattr(outs[1], name)), f"step {step}: {name}"
    with pytest.raises(ValueError, match="pinned"):
        PhysicsViews.from_dict({**dev, "force_matrix_left": phys["force_matrix_left"]}, origins)


def test_global_promotion_over_shards_and_wrapper_outputs():
    """Sharded promotion on the GLOBAL mean (as_fold_stats -> sum over shards -> as_finish_step(global)) equals one
    handle owning all envs; `dones` is terminated | time_out; PhysX-ordered (x,y,z,w) quaternions are accepted."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers

    N, seed, half = 2048, 3, 1024
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    # shard 0 far along, shard 1 at the start: only the global mean crosses the threshold of 12
    st0["curr_target_index"][:half] = 19
    st0["curr_target_index"][half:] = 7
    whole = make_cuda(N, seed)
    shards = [AllstepsMDP(half, device="cuda:0", seed=seed, env_id_offset=r * half) for r in range(2)]
    origins = sc.env_origins.cuda()
    whole.generate_stones(origins)
    keys = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")
    whole.import_state({k: st0[k] for k in keys})
    stw = whole.export_state()
    for r, sh in enumerate(shards):
        sl = slice(r * half, (r + 1) * half)
        sh.import_state({**{k: st0[k][sl] for k in keys}, "steps_pos": stw["steps_pos"][sl],
                         "steps_dphi": stw["steps_dphi"][sl]})
    out = StepBuffers(N, "cuda:0")
    outs = [StepBuffers(half, "cuda:0") for _ in range(2)]
    for step in range(3):
        st = whole.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        dev = {k: v.cuda() for k, v in phys.items()}
        # PhysX order for the shards: x,y,z,w
        dev_xyzw = dict(dev)
        dev_xyzw["root_quat_w"] = dev["root_quat_w"][:, [1, 2, 3, 0]].contiguous()
        whole.step(PhysicsViews.from_dict(dev, origins, sc.body_indices), dev["actions"], out)
        for r, sh in enumerate(shards):
            sl = slice(r * half, (r + 1) * half)
            v = PhysicsViews.from_dict({k: t[sl] for k, t in dev_xyzw.items()}, origins[sl].contiguous(),
                                       sc.body_indices, quat_xyzw=True)
            sh.step(v, dev["actions"][sl], outs[r], finish=False)
            sh.fold_stats()
        g = shards[0].exchange_tensor.clone()
        g[:10] = shards[0].exchange_tensor[:10] + shards[1].exchange_tensor[:10]  # what the NCCL all-reduce produces
        for sh in shards:
            sh.finish_step(g)
        torch.cuda.synchronize()
        for r in range(2):
            sl = slice(r * half, (r + 1) * half)
            for name in ("obs", "reward", "terminated", "time_out", "dones"):
                assert torch.equal(getattr(outs[r], name), getattr(out, name)[sl]), f"step {step} shard {r}: {name}"
            assert torch.equal(shards[r].export_state()["curriculum"], whole.export_state()["curriculum"][sl])
        exact(out.dones, (out.terminated | out.time_out), "dones")
    assert int(whole.export_state()["curriculum"].max()) >= 1, "the global mean (13) must have promoted"


def test_long_replay_100_steps():
    """SURVEY section 7's minimum slice asks for a 100-step replay; run it with everything on (resets, promotion as
    the mean index climbs, per-env levels)."""
    totals, wo, wr = run_replay(2048, 100, seed=123, fall_fraction=0.01, per_env_levels=True)
    assert totals["resets"] > 1000 and totals["advanced"] > 10000
    print(f"100-step replay: {totals}, worst obs rel err {wo:.2e}, reward {wr:.2e}")


def test_config3_size_with_grid_curriculum():
    """BASELINE.json config 3: 65,536 envs with the pitch x yaw grid curriculum (extension), a few steps."""
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao
    from oracle import grid_curriculum as gc

    N, seed, B = 65536, 29, 11
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    grid = gc.GridCurriculum(N, B)
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0),
                            grid=grid, seed=seed)
    mdp = make_cuda(N, seed, grid_bins=B)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    for step in range(3):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, sc.stone_uniforms(step))
        views, keep = to_views(phys, origins, sc.body_indices)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        close(out.reward, o_rew, f"step {step} reward")
        close_obs(out.obs, o_obs, f"step {step} obs")
        bins, att, succ = mdp.grid_state()
        exact(bins, torch.from_numpy(grid.bins.copy()), f"step {step} bins")
        exact(att, torch.from_numpy(grid.attempts.astype(np.int64)), f"step {step} attempts")
        compare_state(mdp, orc, f"step {step}")
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})


def _twin_mdps(N, seed, sc):
    st0 = sc.initial_mdp_state()
    origins = sc.env_origins.cuda()
    mdps = [make_cuda(N, seed) for _ in range(2)]
    for m in mdps:
        m.generate_stones(origins)
        m.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                            "episode_length_buf", "potentials")})
    return mdps, origins, st0


@pytest.mark.parametrize("num_envs", [1001, 4096])
def test_obs_clip_epilogue_equals_the_wrapper_clamp(num_envs):
    """AsStepOut.obs_clip folds RlGamesVecEnvWrapper._process_obs' clamp (isaaclab_rl/rl_games.py:293) into the
    observation write: the clipped buffer is bit-identical to torch.clamp of the raw one, on the fused path and on
    the pass1 / reset / pass2 path; nothing else changes."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    seed, clip = 23, 0.8
    sc = Scenario(num_envs, seed=seed)
    (raw_mdp, clip_mdp), origins, st0 = _twin_mdps(num_envs, seed, sc)
    raw, clipped = StepBuffers(num_envs, "cuda:0"), StepBuffers(num_envs, "cuda:0", obs_clip=clip)
    for step in range(4):
        st = raw_mdp.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        views, keep = to_views(phys, origins, sc.body_indices)
        raw_mdp.step(views, keep["actions"], raw)
        clip_mdp.step(views, keep["actions"], clipped)
        torch.cuda.synchronize()
        assert (raw.obs.abs() > clip).any()
        assert torch.equal(clipped.obs, torch.clamp(raw.obs, -clip, clip)), f"fused step {step}"
        for name in ("reward", "terminated", "time_out", "dones", "reset_joint_pos"):
            assert torch.equal(getattr(raw, name), getattr(clipped, name)), f"fused step {step}: {name}"
    # 3-call path: the clip given to pass1 also applies to the observation rewrite of pass2
    ep_raw = raw_mdp.export_state()["episode_length_buf"].cuda()
    ep_clip = ep_raw.clone()
    for step in range(3):
        st = raw_mdp.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        for mdp, out, ep in ((raw_mdp, raw, ep_raw), (clip_mdp, clipped, ep_clip)):
            views, keep = to_views(phys, origins, sc.body_indices)
            ep += 1
            mdp.pass1(views, keep["actions"], out, episode_length=ep)
            ids = (out.terminated | out.time_out).nonzero().squeeze(-1)
            if len(ids):
                mdp.reset(origins, ids, out, episode_length=ep)
                k = len(ids)
                keep["root_pos_w"][ids] = out.reset_root_state[:k, 0:3]
                keep["root_quat_w"][ids] = out.reset_root_state[:k, 3:7]
                keep["root_lin_vel_w"][ids] = out.reset_root_state[:k, 7:10]
                keep["joint_pos"][ids] = out.reset_joint_pos[:k]
                keep["joint_vel"][ids] = out.reset_joint_vel[:k]
                keep["force_matrix_right"][ids] = 0.0
                keep["force_matrix_left"][ids] = 0.0
                mdp.pass2(views, out)
            else:
                mdp.no_reset()
            torch.cuda.synchronize()
        assert torch.equal(clipped.obs, torch.clamp(raw.obs, -clip, clip)), f"3-call step {step}"
        assert torch.equal(raw.reward, clipped.reward)
    with pytest.raises(Exception, match="obs_clip"):
        bad = StepBuffers(num_envs, "cuda:0", obs_clip=-1.0)
        raw_mdp.step(views, keep["actions"], bad)


def test_nan_inputs_propagate_like_torch():
    """A blown-up physics state (NaN in actions, joint velocities, a foot height, the root quaternion) must show in
    the outputs exactly where it shows in the reference: torch.clamp / torch.minimum hand NaN through (ENV:268,281,337;
    MATH:81-92), comparisons with NaN are false."""
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao

    N, seed = 512, 31
    sc = Scenario(N, seed=seed, fall_fraction=0.0)
    st0 = sc.initial_mdp_state()
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    mdp = make_cuda(N, seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    nan = float("nan")
    for step in range(3):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        phys["actions"][3, 2] = nan
        phys["actions"][200, 20] = nan
        phys["joint_vel"][7, 5] = nan
        phys["joint_pos"][9, 0] = nan
        phys["body_pos_w"][11, sc.body_indices[0], 2] = nan   # right foot height
        phys["body_pos_w"][12, sc.body_indices[1], 2] = nan   # left foot height
        phys["root_quat_w"][13, 1] = nan
        phys["root_lin_vel_w"][14, 0] = nan
        mirror_u, noise_u = sc.reset_uniforms(step)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], mirror_u, noise_u, sc.stone_uniforms(step))
        views, keep = to_views(phys, origins, sc.body_indices)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        for name, got, want in (("obs", out.obs.cpu(), o_obs), ("reward", out.reward.cpu(), o_rew)):
            gn, wn = torch.isnan(got), torch.isnan(want)
            assert torch.equal(gn, wn), (f"step {step}: NaN pattern of {name} differs at "
                                         f"{(gn != wn).nonzero()[:8].tolist()}")
            assert wn.any(), f"step {step}: the reference shows no NaN in {name}; the test would prove nothing"
            ok = ~wn
            if name == "obs":
                close_obs(torch.where(ok, got, torch.zeros_like(got)), torch.where(ok, want, torch.zeros_like(want)),
                          f"step {step} obs")
            else:
                close(got[ok], want[ok], f"step {step} reward")
        st = mdp.export_state()
        exact(st["curr_target_index"], orc.curr_target_index, f"step {step} idx")
        exact(st["target_reach_count"], orc.target_reach_count, f"step {step} count")


def test_extreme_magnitudes_propagate_like_torch():
    """Infinities, values near the top of the float range and denormals in the physics state: overflowing norms
    (inf), inf - inf (NaN), denormal contact forces against the 1e-4 threshold, a zero / denormal quaternion through
    MATH:81-92's normalisation -- masks bit-exact, NaN and inf in the same places, finite values within tolerance.
    (Not covered, documented in as_math.cuh: quotients whose operands overflow or leave 2^+-60 -- a quaternion norm, a
    joint position, a distance of that size: the branch-free divisions give NaN where IEEE division gives 0 or inf;
    observations and rewards only, never a mask.)"""
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao

    N, seed = 512, 37
    sc = Scenario(N, seed=seed, fall_fraction=0.0)
    st0 = sc.initial_mdp_state()
    orc = ao.AllstepsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    mdp = make_cuda(N, seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    install_mdp_state(orc, st0)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    out = StepBuffers(N, "cuda:0")
    inf, big, tiny = float("inf"), 3.0e38, 1.0e-41
    for step in range(3):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        phys["root_lin_vel_w"][3] = torch.tensor([big, big, 0.0])      # the speed overflows to inf: so_fast
        phys["root_lin_vel_w"][4, 1] = -inf
        phys["root_pos_w"][5, 0] = 1.0e15                                # far away, inside 2^+-60
        phys["root_pos_w"][6, 2] = -inf                                  # died; inf - inf further down
        phys["root_quat_w"][7] = torch.tensor([tiny, 0.0, 0.0, 0.0])     # a denormal quaternion: clamp(norm, 1e-9)
        phys["root_quat_w"][8] = 0.0
        phys["root_quat_w"][9] = torch.tensor([1.0e15, -2.0e15, 3.0e15, 1.0e15])  # far from unit, inside 2^+-60
        phys["joint_vel"][10, 3] = inf
        phys["joint_vel"][11, 4] = tiny
        phys["joint_pos"][12, 6] = -1.0e15
        phys["actions"][13, 0] = inf                                     # clamped to 1
        phys["actions"][14, 1] = -inf
        phys["body_pos_w"][15, sc.body_indices[2], 2] = inf              # torso height
        phys["body_pos_w"][16, sc.body_indices[0], :2] = big             # right foot far away
        for k in ("force_matrix_right", "force_matrix_left"):
            idx = orc.curr_target_index
            phys[k][17, 0, idx[17]] = torch.tensor([tiny, tiny, tiny])   # denormal force: no contact
            phys[k][18, 0, idx[18]] = torch.tensor([big, big, big])      # the norm overflows: contact
            phys[k][19, 0, idx[19]] = torch.tensor([0.0, 0.0, inf])
            phys[k][20, 0, idx[20]] = torch.tensor([7.0e-5, 7.0e-5, 0.0])  # |F| = 0.99e-4, just under the threshold
            phys[k][21, 0, idx[21]] = torch.tensor([7.2e-5, 7.2e-5, 0.0])  # just over
        mirror_u, noise_u = sc.reset_uniforms(step)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], mirror_u, noise_u, sc.stone_uniforms(step))
        views, keep = to_views(phys, origins, sc.body_indices)
        mdp.step(views, keep["actions"], out)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        for name, got, want in (("obs", out.obs.cpu(), o_obs), ("reward", out.reward.cpu(), o_rew)):
            gn, wn = torch.isnan(got), torch.isnan(want)
            assert torch.equal(gn, wn), f"step {step}: NaN pattern of {name} differs at {(gn != wn).nonzero()[:8].tolist()}"
            gi, wi = torch.isinf(got), torch.isinf(want)
            assert torch.equal(gi, wi), f"step {step}: inf pattern of {name} differs at {(gi != wi).nonzero()[:8].tolist()}"
            assert torch.equal(got[wi], want[wi]), f"step {step}: sign of an infinity in {name}"
            ok = ~(wn | wi)
            z = torch.zeros_like(got)
            if name == "obs":
                close_obs(torch.where(ok, got, z), torch.where(ok, want, z), f"step {step} obs")
            else:
                close(got[ok], want[ok], f"step {step} reward")
        st = mdp.export_state()
        exact(st["curr_target_index"], orc.curr_target_index, f"step {step} idx")
        exact(st["target_reach_count"], orc.target_reach_count, f"step {step} count")
        exact(st["swing_leg"], orc.swing_leg, f"step {step} leg")


def test_stone_poses_in_physx_view_layout():
    """as_export_stone_poses against a torch restatement of the reference egress: ENV:119-120 builds (N,S,7) w,x,y,z
    poses, RigidObjectCollection.write_object_pose_to_sim (rigid_object_collection.py:295-301) scatters them into
    object_state_w, converts the WHOLE tensor to x,y,z,w, transposes it to object-major (S*N,7)
    (reshape_data_to_view, :650-659) and passes the view ids object*N + env (:675)."""
    N, seed = 777, 5
    sc = Scenario(N, seed=seed)
    mdp = make_cuda(N, seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    steps_pos = mdp.export_state()["steps_pos"]
    S = steps_pos.shape[1]

    def reference_egress(object_state_w, env_ids):
        full = torch.cat((steps_pos, torch.tensor([1.0, 0, 0, 0], device="cuda").repeat(N, S, 1)), dim=-1)
        object_state_w[env_ids[:, None], torch.arange(S, device="cuda"), :7] = full[env_ids].clone()
        poses_xyzw = object_state_w[..., :7].clone()
        poses_xyzw[..., 3:] = poses_xyzw[..., 3:][..., [1, 2, 3, 0]]  # convert_quat(to="xyzw"), MATH:118-155
        view = torch.einsum("ijk -> jik", poses_xyzw).reshape(S * N, 7)
        view_ids = (torch.arange(S, device="cuda").unsqueeze(1) * N + env_ids).flatten()
        return view, view_ids

    # all envs (what __init__ does, ENV:71)
    state = torch.zeros(N, S, 13, device="cuda")
    state[..., 3] = 1.0
    want, want_ids = reference_egress(state, torch.arange(N, device="cuda"))
    got, got_ids = mdp.export_stone_poses()
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert torch.equal(got_ids.long(), want_ids)
    # a subset, unordered, into a persistent buffer: other rows stay as they are
    ids = torch.tensor([5, 700, 3, 64, 776, 0], device="cuda")
    buf = torch.full((S * N, 7), -7.0, device="cuda")
    got, got_ids = mdp.export_stone_poses(ids, buf)
    torch.cuda.synchronize()
    assert torch.equal(got_ids.long(), (torch.arange(S, device="cuda").unsqueeze(1) * N + ids).flatten())
    assert torch.equal(got[got_ids.long()], want[got_ids.long()])
    untouched = torch.ones(S * N, dtype=torch.bool, device="cuda")
    untouched[got_ids.long()] = False
    assert (got[untouched] == -7.0).all()
    _, none_ids = mdp.export_stone_poses(torch.empty(0, dtype=torch.int64, device="cuda"), buf)
    assert none_ids.numel() == 0


def test_peer_exchange_world_of_one_equals_the_plain_step():
    """The peer-memory route with a single rank (the exchange kernel stores to and reads from its own buffer) must
    change nothing: same outputs, same levels (promotions included), global counters == local counters."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    N, seed = 3000, 19
    sc = Scenario(N, seed=seed)
    (plain, peer), origins, st0 = _twin_mdps(N, seed, sc)
    hi = torch.randint(11, 20, (N,), generator=sc.gen)
    for m in (plain, peer):
        m.import_state({"curr_target_index": hi})
    peer.connect_self()
    outs = [StepBuffers(N, "cuda:0"), StepBuffers(N, "cuda:0")]
    levels = set()
    for step in range(10):
        st = plain.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        views, keep = to_views(phys, origins, sc.body_indices)
        plain.step(views, keep["actions"], outs[0])
        peer.step(views, keep["actions"], outs[1])
        torch.cuda.synchronize()
        for name in ("obs", "reward", "terminated", "time_out", "dones", "reset_joint_pos"):
            assert torch.equal(getattr(outs[0], name), getattr(outs[1], name)), f"step {step}: {name}"
        a, b = plain.export_state(), peer.export_state()
        for k in a:
            assert torch.equal(a[k], b[k]), f"step {step}: state {k}"
        assert torch.equal(peer.global_stats_tensor[:10], peer.stats_tensor[:10])
        assert plain.read_stats() == peer.read_stats()
        levels.add(int(b["curriculum"].max()))
    assert len(levels) > 1, "no promotion happened"
    assert peer.peer_status() == {"world": 1, "rank": 0, "timeouts": 0}
    # quiet steps: nobody resets anywhere, so the exchanging CTA leaves the step open and the fix-up kernel redoes it
    # without pass 2 on the exchanged record -- and with the grid curriculum the exchange runs as a kernel of its own
    for kw, n_quiet in ((dict(), 40), (dict(grid_bins=4), 40)):
        scq = Scenario(n_quiet, seed=seed + 1, fall_fraction=0.0)
        originsq = scq.env_origins.cuda()
        twins = [make_cuda(n_quiet, seed, **kw) for _ in range(2)]
        st0q = scq.initial_mdp_state()
        for m in twins:
            m.generate_stones(originsq)
            m.import_state({k: st0q[k] for k in ("curr_target_index", "swing_leg", "target_reach_count", "potentials")})
        twins[1].connect_self()
        quiet = 0
        for step in range(8):
            st = twins[0].export_state()
            phys = scq.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
            phys["root_lin_vel_w"] *= 0.1
            views, keep = to_views(phys, originsq, scq.body_indices)
            o = [StepBuffers(n_quiet, "cuda:0"), StepBuffers(n_quiet, "cuda:0")]
            twins[0].step(views, keep["actions"], o[0])
            twins[1].step(views, keep["actions"], o[1])
            torch.cuda.synchronize()
            quiet += int(int(o[0].n_reset.item()) == 0)
            for name in ("obs", "reward", "terminated", "time_out"):
                assert torch.equal(getattr(o[0], name), getattr(o[1], name)), f"{kw} quiet step {step}: {name}"
            a, b = twins[0].export_state(), twins[1].export_state()
            for k in a:
                assert torch.equal(a[k], b[k]), f"{kw} quiet step {step}: state {k}"
        assert quiet > 0
        assert twins[1].peer_status()["timeouts"] == 0


def test_programmatic_launch_chain_changes_nothing(monkeypatch):
    """gather -> step -> finish are chained by programmatic dependent launch (each kernel starts under the tail of the
    one before and waits with griddepcontrol.wait before it reads what that one wrote).  Against a handle created
    with ALLSTEPS_PDL=0 (plain stream order) every output and the whole MDP state must be bit-identical."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    N, seed = (1 << 17) + 37, 47
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    origins = sc.env_origins.cuda()
    monkeypatch.setenv("ALLSTEPS_PDL", "0")
    plain = make_cuda(N, seed)
    monkeypatch.delenv("ALLSTEPS_PDL")
    chained = make_cuda(N, seed)
    for m in (plain, chained):
        m.generate_stones(origins)
        m.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                            "episode_length_buf", "potentials")})
    outs = [StepBuffers(N, "cuda:0"), StepBuffers(N, "cuda:0")]
    for step in range(4):
        st = plain.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        views, keep = to_views(phys, origins, sc.body_indices)
        for o in outs:
            o.obs.fill_(float("nan"))
        plain.step(views, keep["actions"], outs[0])
        chained.step(views, keep["actions"], outs[1])
        torch.cuda.synchronize()
        assert not torch.isnan(outs[1].obs).any()
        for name in ("obs", "reward", "terminated", "time_out", "dones", "reset_root_state", "reset_joint_pos"):
            assert torch.equal(getattr(outs[0], name), getattr(outs[1], name)), f"step {step}: {name}"
        a, b = plain.export_state(), chained.export_state()
        for k in a:
            assert torch.equal(a[k], b[k]), f"step {step}: state {k}"


def test_resume_from_a_checkpoint_is_bit_identical():
    """SURVEY section 5: state_dict() / load_state_dict() incl. the Philox position, the pending promotion and the
    grid-curriculum state -- a run resumed in a FRESH handle continues bit for bit like the uninterrupted one."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers

    for kw in (dict(), dict(grid_bins=5), dict(intended_regen=True)):
        N, seed = 3000, 41
        sc = Scenario(N, seed=seed, fall_fraction=0.2)
        origins = sc.env_origins.cuda()
        st0 = sc.initial_mdp_state()
        st0["curr_target_index"] = torch.randint(11, 20, (N,), generator=sc.gen)  # promotions will happen

        def fresh():
            m = AllstepsMDP(N, device="cuda:0", seed=seed, **kw)
            m.generate_stones(origins)
            return m

        mdp = fresh()
        mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                              "episode_length_buf", "potentials")})
        out = StepBuffers(N, "cuda:0")

        def physics_for(m):
            st = m.export_state()
            phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
            d = {k: v.cuda() for k, v in phys.items()}
            return PhysicsViews.from_dict(d, origins, sc.body_indices), d

        for _ in range(5):
            v, d = physics_for(mdp)
            mdp.step(v, d["actions"], out)
        ckpt = mdp.state_dict()
        assert int(ckpt["meta"][1]) == N
        tail = [physics_for(mdp)]
        record = []
        for i in range(6):
            v, d = tail[-1]
            mdp.step(v, d["actions"], out)
            torch.cuda.synchronize()
            record.append({k: getattr(out, k).clone() for k in ("obs", "reward", "terminated", "time_out",
                                                                "reset_joint_pos", "reset_root_state")})
            record[-1]["state"] = mdp.export_state()
            tail.append(physics_for(mdp))
        levels = int(record[-1]["state"]["curriculum"].max())
        resumed = fresh()
        with pytest.raises(ValueError):
            AllstepsMDP(N, device="cuda:0", seed=seed + 1, **kw).load_state_dict(ckpt)
        resumed.load_state_dict(ckpt)
        out2 = StepBuffers(N, "cuda:0")
        for i in range(6):
            v, d = tail[i]
            resumed.step(v, d["actions"], out2)
            torch.cuda.synchronize()
            for k in ("obs", "reward", "terminated", "time_out"):
                assert torch.equal(getattr(out2, k), record[i][k]), f"{kw} step {i}: {k} differs after the resume"
            ids = record[i]["terminated"] | record[i]["time_out"]
            assert torch.equal(out2.reset_joint_pos[ids], record[i]["reset_joint_pos"][ids])
            st = resumed.export_state()
            for k, ref in record[i]["state"].items():
                assert torch.equal(st[k], ref), f"{kw} step {i}: state {k} differs after the resume"
        if not kw:
            assert levels > 0, "no promotion in the replay: the pending-promotion part of the checkpoint went untested"
        if kw.get("grid_bins"):
            a, b = mdp.grid_state(), resumed.grid_state()
            for x, y in zip(a, b):
                assert torch.equal(x, y)
        # an in-place rewind of a live handle (what bench.py does to keep its input sets on the state they were made for)
        snap = mdp.snapshot(include_stones=True)
        before = mdp.export_state()
        v, d = tail[-1]
        mdp.step(v, d["actions"], out)
        mdp.restore(snap, include_stones=True)
        after = mdp.export_state()
        for k in before:
            assert torch.equal(before[k], after[k]), k


@pytest.mark.parametrize("N,fall", [(3000, 0.03), (40, 0.0), ((1 << 17) + 5, 0.02)])
def test_three_call_path_with_the_device_side_reset_list(N, fall):
    """as_reset(env_ids = NULL): the envs pass 1 flagged come from the id list it compacted on the device -- no
    `.nonzero()` -- and as_step_pass2 decides on the device whether anything reset at all.  Must equal the flow with the
    host's id tensor (DRL:359) bit for bit, in busy and in quiet steps."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    seed = 71
    sc = Scenario(N, seed=seed, fall_fraction=fall)
    (host_mdp, dev_mdp), origins, st0 = _twin_mdps(N, seed, sc)
    out_h, out_d = StepBuffers(N, "cuda:0"), StepBuffers(N, "cuda:0")
    ep_h = st0["episode_length_buf"].cuda().clone()
    ep_d = ep_h.clone()

    def writes(keep, ids, out, k):
        keep["root_pos_w"][ids] = out.reset_root_state[:k, 0:3]
        keep["root_quat_w"][ids] = out.reset_root_state[:k, 3:7]
        keep["root_lin_vel_w"][ids] = out.reset_root_state[:k, 7:10]
        keep["joint_pos"][ids] = out.reset_joint_pos[:k]
        keep["joint_vel"][ids] = out.reset_joint_vel[:k]
        keep["force_matrix_right"][ids] = 0.0
        keep["force_matrix_left"][ids] = 0.0

    quiet = busy = 0
    for step in range(8):
        st = host_mdp.export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        vh, kh = to_views(phys, origins, sc.body_indices)
        vd, kd = to_views(phys, origins, sc.body_indices)
        ep_h += 1
        ep_d += 1
        host_mdp.pass1(vh, kh["actions"], out_h, episode_length=ep_h)
        ids = out_h.dones.nonzero().squeeze(-1)
        if len(ids):
            host_mdp.reset(origins, ids, out_h, episode_length=ep_h)
            writes(kh, ids, out_h, len(ids))
            host_mdp.pass2(vh, out_h)
            busy += 1
        else:
            host_mdp.no_reset()
            quiet += 1
        dev_mdp.pass1(vd, kd["actions"], out_d, episode_length=ep_d)
        dev_mdp.reset(origins, None, out_d, episode_length=ep_d)
        n = int(out_d.n_reset.item())          # (the test plays PhysX: it needs the rows on the host side)
        assert n == len(ids)
        ids_d = out_d.reset_ids[:n].long()
        assert torch.equal(ids_d.sort().values, ids)
        writes(kd, ids_d, out_d, n)
        dev_mdp.pass2(vd, out_d)
        torch.cuda.synchronize()
        for name in ("obs", "reward", "terminated", "time_out", "dones"):
            assert torch.equal(getattr(out_h, name), getattr(out_d, name)), f"step {step}: {name}"
        assert torch.equal(ep_h, ep_d)
        a, b = host_mdp.export_state(), dev_mdp.export_state()
        for k in a:
            assert torch.equal(a[k], b[k]), f"step {step}: state {k}"
    assert (quiet > 0) if fall == 0.0 else (busy > 0)


def test_port_run_as_eager_cuda_torch_agrees_within_tolerance():
    """The parity target of the bit-exact claims is the reference on CPU torch (the only reference that can be executed
    and recorded: tests/golden).  Isaac Lab runs the same ops as eager CUDA torch, whose kernels may round a few of
    them differently (division by a Python scalar as a multiplication by its reciprocal, reduction order of
    vector_norm / cumsum).  This runs the port with CUDA tensors next to the kernels: floating point stays inside the
    1e-5 tolerance, and no mask or index differs on this replay."""
    from allsteps_isaaclab_b200.mdp import StepBuffers
    from oracle import allsteps_oracle as ao

    N, seed = 4096, 83
    sc = Scenario(N, seed=seed)
    st0 = sc.initial_mdp_state()
    mdp = make_cuda(N, seed)
    origins = sc.env_origins.cuda()
    mdp.generate_stones(origins)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    with torch.device("cuda:0"):
        orc = ao.AllstepsOracle(sc.cfg, N, origins, sc.joint_limits.cuda(), sc.body_indices, sc.stone_uniforms(0).cuda())
        install_mdp_state(orc, {k: v.cuda() for k, v in st0.items()})
        mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
        out = StepBuffers(N, "cuda:0")
        mask_diffs = 0
        for step in range(6):
            phys = sc.physics(orc.steps_pos.cpu(), orc.curr_target_index.cpu(), orc.swing_leg.cpu())
            m, n = sc.reset_uniforms(step)
            d = {k: v.cuda() for k, v in phys.items()}
            o_obs, o_rew, o_term, o_to, _ = orc.step(d, d["actions"], m.cuda(), n.cuda(), None)
            views, keep = to_views(phys, origins, sc.body_indices)
            mdp.step(views, keep["actions"], out)
            torch.cuda.synchronize()
            mask_diffs += int((out.terminated != o_term).sum()) + int((out.time_out != o_to).sum())
            st = mdp.export_state()
            mask_diffs += int((st["curr_target_index"] != orc.curr_target_index).sum())
            same = (out.terminated == o_term) & (out.time_out == o_to)
            close(out.reward[same], o_rew[same], f"step {step} reward vs CUDA torch")
            close_obs(out.obs[same], o_obs[same], f"step {step} obs vs CUDA torch")
            mdp.import_state({k: getattr(orc, k) for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                                           "potentials")})
        assert mask_diffs == 0, f"{mask_diffs} mask / index differences against the port run on CUDA torch"
