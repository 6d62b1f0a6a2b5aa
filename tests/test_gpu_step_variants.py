"""Every `k_step` instantiation against the oracle: reward term by term, statistic by statistic.

Each case of `step_variants.CASES` proves with the CUDA profiler which instantiations its step launched, then replays
a few steps against `TermsOracle`: obs, reward, masks, reset rows and state as in tests/test_gpu_parity.py, the ten
reward terms column by column on all rows (generic instantiations), and every `AsStats` field.  Bar: integer / mask
outputs and statistics exact; fp32 within 1e-5 relative; `sum_reward` (fp32 atomics, order not fixed) within
1e-5 * sum(max(1, |r|)) of the float64 sum of the oracle's rewards.
"""
from __future__ import annotations

import math

import pytest
import torch

import edge_scenario as edge
import step_variants as sv
from allsteps_isaaclab_b200 import synthetic as syn
from scenario import Scenario, install_mdp_state
from terms_oracle import STAT_FIELDS, TermsOracle

pytestmark = pytest.mark.gpu

RTOL = 1e-5
OBS_CLIP = 3.0
QUIET_STEP = 1  # the step of every replay in which no env resets (fix-up / no_reset routes)


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


def to_views(phys, env_origins_cuda, body_rows, layout="contiguous", quat_xyzw=False):
    """Move one synthetic physics dict to the GPU in a chosen memory layout (quat_xyzw: PhysX' quaternion order)."""
    from allsteps_isaaclab_b200.mdp import PhysicsViews

    d = {k: v.cuda() for k, v in phys.items()}
    if quat_xyzw:
        d["root_quat_w"] = d["root_quat_w"][:, [1, 2, 3, 0]].contiguous()
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
    elif layout == "pinned_contact":
        for k in ("force_matrix_right", "force_matrix_left"):
            d[k] = phys[k].pin_memory()
    return PhysicsViews.from_dict(d, env_origins_cuda, body_rows, quat_xyzw=quat_xyzw), d


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


def compare_stats(stats, orc, what, fields=STAT_FIELDS):
    want = orc.stats
    bad = {k: (stats[k], want[k]) for k in fields if stats[k] != want[k]}
    assert not bad, f"{what}: AsStats (kernel, oracle) differ: {bad}"
    # fp32 atomics in no fixed order: a dropped or doubled warp / tile is far outside this bound
    bound = 1e-5 * float(orc.last_reward.double().abs().clamp(min=1.0).sum())
    assert abs(stats["sum_reward"] - orc.reward_sum) <= bound, \
        f"{what}: sum_reward {stats['sum_reward']} vs {orc.reward_sum} (bound {bound:.3g})"


def launched_step_kernels(launch):
    """The (MODE, EXACT, FULL, FAST, PACKED, PRE) of every k_step that `launch()` ran, from a CUDA profiler trace."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        launch()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert names, "the CUDA profiler recorded no kernel: the instantiation check would be empty"
    found = [sv.parse_kernel_name(n) for n in names if "k_step<" in n]
    assert all(f is not None for f in found), f"unparsed k_step names: {sorted(n for n in names if 'k_step<' in n)}"
    return set(found), names


def expected_kernels(case):
    by_row = sv.rows_by_number(sv.parse_step_variants())
    return {by_row[r].template for r in case.rows}


def exact_div_cfg():
    from allsteps_isaaclab_b200.config import AllstepsCfg

    class Cfg(AllstepsCfg):
        def joint_limits_rad(self):
            lim = list(super().joint_limits_rad())
            lim[9] = (0.0, 1.9999998807907104)  # fp32 0x3fffffff: an all-ones significand
            return lim

    return Cfg()


def quiet(phys):
    """No env terminates in this state: velocities below max_root_speed (the synthetic state has no falls when its
    fall fraction is 0)."""
    v = phys["root_lin_vel_w"]
    phys["root_lin_vel_w"] = v * (4.0 / torch.linalg.vector_norm(v, dim=-1, keepdim=True)).clamp(max=1.0)
    return phys


def physics(sc, orc, step):
    if step != QUIET_STEP:
        return sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    return quiet(syn.random_physics_state(sc.cfg, orc.steps_pos, orc.curr_target_index, orc.swing_leg, sc.gen,
                                          num_bodies=sc.num_bodies, body_indices=sc.body_indices, fall_fraction=0.0))


class Replay:
    """Oracle + handle from one seeded state.  Episode lengths are kept away from the time-out except for a few envs
    that time out in steps 0 and 2, so that step QUIET_STEP resets nobody."""

    def __init__(self, num_envs, seed, cfg=None, full_bodies=False):
        self.sc = sc = Scenario(num_envs, seed=seed, cfg=cfg, full_bodies=full_bodies)
        st0 = sc.initial_mdp_state()
        ep = st0["episode_length_buf"] % 880
        ep[::97] = 898   # time out in step 0
        ep[5::89] = 896  # time out in step 2
        st0["episode_length_buf"] = ep
        self.st0 = st0
        self.orc = TermsOracle(sc.cfg, num_envs, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
        self.origins = sc.env_origins.cuda()
        install_mdp_state(self.orc, st0)
        self.mdps = []
        self.new_handle()

    def new_handle(self):
        from allsteps_isaaclab_b200.mdp import AllstepsMDP

        sc, st0 = self.sc, self.st0
        mdp = AllstepsMDP(sc.N, device="cuda:0", cfg=sc.cfg, seed=sc.seed)
        mdp.generate_stones(self.origins)
        mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                              "episode_length_buf", "potentials")})
        mdp.import_state({"steps_pos": self.orc.steps_pos, "steps_dphi": self.orc.steps_dphi})
        self.mdps.append(mdp)
        return mdp


def physx_writes(keep, ids, out, k, quat_xyzw=False):
    """What `_reset_idx` hands to PhysX lands in the data views (ART:316-489); scene.reset zeroes the contacts."""
    q = out.reset_root_state[:k, 3:7]
    keep["root_pos_w"][ids] = out.reset_root_state[:k, 0:3]
    keep["root_quat_w"][ids] = q[:, [1, 2, 3, 0]] if quat_xyzw else q
    keep["root_lin_vel_w"][ids] = out.reset_root_state[:k, 7:10]
    keep["joint_pos"][ids] = out.reset_joint_pos[:k]
    keep["joint_vel"][ids] = out.reset_joint_vel[:k]
    keep["force_matrix_right"][ids] = 0.0
    keep["force_matrix_left"][ids] = 0.0


def three_call(mdp, views, keep, out, ep_len, origins, device_list=False, quat_xyzw=False):
    """pass1 -> reset -> PhysX writes -> pass2, or pass1 -> no_reset when nothing reset (DRL:359-360)."""
    mdp.pass1(views, keep["actions"], out, episode_length=ep_len)
    if device_list:
        mdp.reset(origins, None, out, episode_length=ep_len)
        n = int(out.n_reset.item())
        ids = out.reset_ids[:n].long()
        physx_writes(keep, ids, out, n, quat_xyzw)
        mdp.pass2(views, out)
        return ids.sort().values
    ids = out.dones.nonzero().squeeze(-1)
    if len(ids):
        mdp.reset(origins, ids, out, episode_length=ep_len)
        physx_writes(keep, ids, out, len(ids), quat_xyzw)
        mdp.pass2(views, out)
    else:
        mdp.no_reset()
    return ids


def check_outputs(out, orc, o_obs, o_rew, o_term, o_to, o_ids, what, obs_clip=0.0, terms=False, final_obs=False,
                  host_ids=None):
    exact(out.terminated, o_term, f"{what} terminated")
    exact(out.time_out, o_to, f"{what} time_out")
    close(out.reward, o_rew, f"{what} reward")
    want_obs = o_obs.clamp(-obs_clip, obs_clip) if obs_clip else o_obs
    close_obs(out.obs, want_obs, f"{what} obs")
    if terms:
        for c in range(10):
            close(out.reward_terms[:, c], orc.terms[:, c], f"{what} reward term {c}")
            exact(out.reward_terms[:, c] != 0, orc.terms[:, c] != 0, f"{what} reward term {c} zero mask")
    if final_obs and len(o_ids):
        fin = orc.final_obs.clamp(-obs_clip, obs_clip) if obs_clip else orc.final_obs
        close_obs(out.final_obs[o_ids.cuda()], fin[o_ids], f"{what} final_obs")
    if host_ids is None:  # fused: the step wrote the reset list and rows
        n = int(out.n_reset.item())
        assert n == len(o_ids), f"{what}: n_reset {n} vs {len(o_ids)}"
        ids = out.reset_ids[:n].long().sort().values
        exact(ids, o_ids, f"{what} reset ids")
    else:
        exact(host_ids, o_ids, f"{what} reset ids")
        ids = host_ids
    if len(o_ids):
        w = orc.reset_writes
        k = len(o_ids)
        rows = ids.cuda() if host_ids is None else torch.arange(k, device="cuda")
        close(out.reset_root_state[rows], torch.cat((w["root_pose"], w["root_velocity"]), -1), f"{what} reset root")
        close(out.reset_joint_pos[rows], w["joint_pos"], f"{what} reset joint_pos")
        close(out.reset_joint_vel[rows], w["joint_vel"], f"{what} reset joint_vel")


@pytest.mark.parametrize("case", sv.CASES, ids=lambda c: c.name)
def test_step_variant_against_the_oracle(case):
    from allsteps_isaaclab_b200.mdp import StepBuffers

    cfg = exact_div_cfg() if case.exact_div else None
    rp = Replay(case.num_envs, seed=300 + sv.CASES.index(case), cfg=cfg, full_bodies=case.layout == "isaac")
    sc, orc, mdp, origins = rp.sc, rp.orc, rp.mdps[0], rp.origins
    xyzw = "quat_xyzw" in case.outputs
    clip = OBS_CLIP if "obs_clip" in case.outputs else 0.0
    out = StepBuffers(case.num_envs, "cuda:0", reward_terms="reward_terms" in case.outputs, obs_clip=clip,
                      final_obs="final_obs" in case.outputs)
    want = expected_kernels(case)
    if case.mode == "pass2":
        return pass2_outside_a_step(case, rp, out, want)
    ep_len = rp.st0["episode_length_buf"].cuda()
    totals = dict(resets=0, advanced=0)
    for step in range(4):
        phys = physics(sc, orc, step)
        m, n = sc.reset_uniforms(step if case.mode == "fused" else step + 1)  # (pass 1 advances the step counter)
        o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, None)
        views, keep = to_views(phys, origins, sc.body_indices, case.layout, quat_xyzw=xyzw)
        host_ids = None
        if case.mode == "fused":
            launch = lambda: mdp.step(views, keep["actions"], out)  # noqa: E731
        else:
            ep_len += 1  # DRL:351
            res = {}
            launch = lambda: res.setdefault("ids", three_call(mdp, views, keep, out, ep_len, origins,  # noqa: E731
                                                              quat_xyzw=xyzw))
        if step == 0:
            got, names = launched_step_kernels(launch)
            assert got == want, f"{case.name}: launched {sorted(got)}, expected rows {case.rows} = {sorted(want)}"
        else:
            launch()
        torch.cuda.synchronize()
        if case.mode != "fused":
            host_ids = res["ids"]
            exact(ep_len, orc.episode_length_buf, f"step {step} episode_length")
        what = f"{case.name} step {step}"
        assert (len(o_ids) == 0) == (step == QUIET_STEP), f"{what}: {len(o_ids)} resets"
        check_outputs(out, orc, o_obs, o_rew, o_term, o_to, o_ids, what, obs_clip=clip,
                      terms="reward_terms" in case.outputs, final_obs="final_obs" in case.outputs,
                      host_ids=host_ids)
        compare_state(mdp, orc, what)
        compare_stats(mdp.read_stats(), orc, what)
        totals["resets"] += len(o_ids)
        totals["advanced"] += orc.stats["n_advanced"]
    assert totals["resets"] > 0 and totals["advanced"] > 0


def pass2_outside_a_step(case, rp, out, want):
    """DirectRLEnv.reset() (DRL:256-279): `_reset_idx(all envs)` -> PhysX writes -> ENV:567, with no pass 1 open; then
    a fused step from there."""
    sc, orc, mdp, origins = rp.sc, rp.orc, rp.mdps[0], rp.origins
    N = sc.N
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    ids = torch.arange(N)
    sum_index = int(orc.curr_target_index.sum())
    m, n = sc.reset_uniforms(1)  # (the reset outside a step advances the Philox step counter first)
    orc.load_physics(phys)
    orc.reset_rows(ids, m, n, None)
    views, keep = to_views(phys, origins, sc.body_indices, case.layout)
    mdp.reset(origins, ids.cuda(), out)
    physx_writes(keep, ids.cuda(), out, N)
    got, _ = launched_step_kernels(lambda: mdp.pass2(views, out))
    assert got == want, f"{case.name}: launched {sorted(got)}, expected rows {case.rows} = {sorted(want)}"
    torch.cuda.synchronize()
    close_obs(out.obs, orc.observations(), "pass 2 obs")
    compare_state(mdp, orc, "after the reset")
    stats = mdp.read_stats()
    # the reset outside a step records what the promotion rule of ENV:471 read, and the new step counter
    assert stats["n_envs"] == N and stats["sum_target_index"] == sum_index and stats["step_counter"] == 1, stats
    # ... then the first step of the episode
    orc.step_index = 1
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    m, n = sc.reset_uniforms(1)
    o_obs, o_rew, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, None)
    views, keep = to_views(phys, origins, sc.body_indices, case.layout)
    mdp.step(views, keep["actions"], out)
    torch.cuda.synchronize()
    check_outputs(out, orc, o_obs, o_rew, o_term, o_to, o_ids, "first step", terms=True)
    compare_state(mdp, orc, "first step")
    compare_stats(mdp.read_stats(), orc, "first step")


@pytest.mark.parametrize("num_envs", [65536, 4096 + 7])
def test_fused_and_three_call_statistics_agree(num_envs):
    """The same steps through the fused step and through the 3-call path (host ids; device-side list) from one
    state: every AsStats field but sum_reward is equal, and equal to the oracle's -- in steps with resets and in a step
    without (fused: the fix-up discards pass 2; 3-call: as_step_no_reset, or k_pass2_commit finding an empty list)."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    rp = Replay(num_envs, seed=77)
    fused = rp.mdps[0]
    host, dev = rp.new_handle(), rp.new_handle()
    sc, orc, origins = rp.sc, rp.orc, rp.origins
    outs = [StepBuffers(num_envs, "cuda:0") for _ in range(3)]
    ep = [rp.st0["episode_length_buf"].cuda() for _ in range(2)]
    fields = list(STAT_FIELDS)
    for step in range(3):
        phys = physics(sc, orc, step)
        # the fused handle draws at its step counter; the 3-call handles' resets at the counter after pass 1 --
        # the same rows only when no env resets, so the oracle follows the fused handle and the 3-call handles are
        # compared field by field
        m, n = sc.reset_uniforms(step)
        orc.step(phys, phys["actions"], m, n, None)
        v0, k0 = to_views(phys, origins, sc.body_indices)
        fused.step(v0, k0["actions"], outs[0])
        for i, (mdp, device_list) in enumerate(((host, False), (dev, True))):
            v, k = to_views(phys, origins, sc.body_indices)
            ep[i] += 1
            three_call(mdp, v, k, outs[1 + i], ep[i], origins, device_list=device_list)
        torch.cuda.synchronize()
        what = f"N {num_envs} step {step}"
        s_f, s_h, s_d = fused.read_stats(), host.read_stats(), dev.read_stats()
        compare_stats(s_f, orc, f"{what} fused")
        for name, s in (("host ids", s_h), ("device list", s_d)):
            bad = {f: (s[f], s_f[f]) for f in fields if s[f] != s_f[f]}
            assert not bad, f"{what}: 3-call ({name}) vs fused AsStats differ: {bad}"
        assert (orc.stats["n_reset"] == 0) == (step == QUIET_STEP)
        if step != QUIET_STEP:
            assert int(orc.advanced2.sum()) > 0, "no pass-2 advance: the step does not tell the paths apart"
        # the state after the step: from here on all three handles continue from the oracle's
        for mdp in (host, dev):
            mdp.import_state({k: getattr(orc, k) for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                                           "potentials", "curriculum")})
        for i in range(2):
            ep[i].copy_(orc.episode_length_buf)


@pytest.mark.parametrize("route", ["fused-fast", "fused-generic", "three-call"])
def test_edge_scenario(route):
    """The edge scenario (tests/edge_scenario.py): decisions on their thresholds with exact operands, in a full tile
    and in a ragged one.  Every mask and the exact reward terms must equal the oracle's bit for bit."""
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers

    es = edge.EdgeScenario(copies=(0, 256))
    N = es.N
    orc = TermsOracle(es.cfg, N, es.env_origins, es.joint_limits, es.body_indices, None)
    es.install(orc)
    mdp = AllstepsMDP(N, device="cuda:0", cfg=es.cfg, seed=es.seed)
    mdp.import_state({k: es.state[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                               "episode_length_buf", "curriculum", "potentials")})
    mdp.import_state({"steps_pos": es.steps_pos, "steps_dphi": es.steps_dphi})
    generic = route != "fused-fast"
    out = StepBuffers(N, "cuda:0", reward_terms=generic)
    m, n = es.reset_uniforms(0 if route != "three-call" else 1)
    o_obs, o_rew, o_term, o_to, o_ids = orc.step(es.phys, es.phys["actions"], m, n, None)
    origins = es.env_origins.cuda()
    views, keep = to_views(es.phys, origins, es.body_indices)
    host_ids = None
    if route == "three-call":
        ep_len = es.state["episode_length_buf"].cuda() + 1
        host_ids = three_call(mdp, views, keep, out, ep_len, origins)
    else:
        mdp.step(views, keep["actions"], out)
    torch.cuda.synchronize()
    check_outputs(out, orc, o_obs, o_rew, o_term, o_to, o_ids, route, terms=generic, host_ids=host_ids)
    compare_state(mdp, orc, route)
    compare_stats(mdp.read_stats(), orc, route)
    st = mdp.export_state()
    # (masks: terminated / time_out above, fell / so_fast / died in the statistics; pressed: the contact columns;
    # reached: the reach counts; clamp, limit, speed, bonus: the exact terms)
    exact(out.obs[:, 48:50], orc.observations()[:, 48:50], f"{route} foot contacts")
    if generic:
        t = out.reward_terms.cpu()
        for c in edge.EXACT_TERM_COLUMNS:
            exact(t[:, c], orc.terms[:, c], f"{route} reward term {c}")
        for c in range(10):
            exact(t[:, c] != 0, orc.terms[:, c] != 0, f"{route} reward term {c} zero mask")
    else:
        exact(out.reward[~o_term.cuda()].cpu() != 0, o_rew[~o_term] != 0, f"{route} reward zero mask")
    exact(st["target_reach_count"], orc.target_reach_count, f"{route} reach counts")
