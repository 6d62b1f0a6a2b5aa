"""GPU: AsStepOut.final_obs -- the observation of the state an env's episode ended in, written by the step kernels for
the envs that reset -- against the oracle's `final_obs` (the row `_get_observations()` returns between `_get_rewards`
and `_reset_idx`), on the fused step and on the 3-call path.  Switching the output on must change nothing else."""
from __future__ import annotations

import types

import pytest
import torch

from final_obs_oracle import FinalObsOracle
from scenario import Scenario, install_mdp_state
from test_gpu_parity import close_obs, exact, make_cuda, to_views

pytestmark = pytest.mark.gpu

# prefill of the final-observation buffers: a NaN payload no kernel produces, so an untouched row is recognisable
PREFILL = 0x7FC0_0D0E
OUTPUTS = ("obs", "reward", "terminated", "time_out", "dones", "reset_root_state", "reset_joint_pos",
           "reset_joint_vel")
STATE_KEYS = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")


def bits(t: torch.Tensor) -> torch.Tensor:
    """The bytes of a tensor, so that equal NaNs compare equal."""
    return t.detach().contiguous().view(torch.uint8).cpu()


def same_bits(a: torch.Tensor, b: torch.Tensor, what: str):
    assert torch.equal(bits(a), bits(b)), what


def final_buffers(N, **kw):
    from allsteps_isaaclab_b200.mdp import StepBuffers

    out = StepBuffers(N, "cuda:0", final_obs=True, **kw)
    out.final_obs.view(torch.int32).fill_(PREFILL)
    return out


def expected_final(orc, clip):
    f = orc.final_obs
    return torch.clamp(f, -clip, clip) if clip > 0 else f


def setup(N, seed, fall, full_bodies=False, n_mdps=2):
    """Oracle + `n_mdps` handles on the same seeded state; every 7th env is two steps from its time-out."""
    sc = Scenario(N, seed=seed, fall_fraction=fall, full_bodies=full_bodies)
    st0 = sc.initial_mdp_state()
    st0["episode_length_buf"][::7] = 897
    orc = FinalObsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    install_mdp_state(orc, st0)
    origins = sc.env_origins.cuda()
    mdps = [make_cuda(N, seed) for _ in range(n_mdps)]
    for m in mdps:
        m.import_state({k: st0[k] for k in STATE_KEYS})
        m.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi})
    return sc, orc, origins, mdps


def check_final_rows(out, expect, ids, o_final, what):
    """Rows of `ids` equal the oracle's; every other row is what it was before the step (`expect`, updated here)."""
    if len(ids):
        close_obs(out.final_obs[ids], o_final[ids], f"{what} final_obs of the envs that reset")
        expect[ids] = out.final_obs[ids].cpu()
    same_bits(out.final_obs, expect, f"{what}: final_obs rows of envs that did not reset were written")


def compare_twins(a, b, out_a, out_b, what, compact=None):
    """`compact`: the reset rows are compact (3-call path); "device_list": in the order of the device-side id list,
    which atomics fill in no fixed order -- compared sorted by env id."""
    for name in OUTPUTS:
        x, y = getattr(out_a, name), getattr(out_b, name)
        if compact and name.startswith("reset_"):
            n = int(out_a.n_reset.item()) if compact == "device_list" else int(out_a.dones.sum())
            if compact == "device_list":
                x = x[:n][out_a.reset_ids[:n].argsort()]
                y = y[:n][out_b.reset_ids[:n].argsort()]
            x, y = x[:n], y[:n]
        same_bits(x, y, f"{what}: {name} differs with final_obs on")
    sa, sb = a.export_state(), b.export_state()
    for k in sa:
        same_bits(sa[k], sb[k], f"{what}: state {k} differs with final_obs on")
    ra, rb = a.read_stats(), b.read_stats()
    # (the reward sum is accumulated by float atomics of all CTAs, in no fixed order: equal up to rounding)
    sa_r, sb_r = ra.pop("sum_reward"), rb.pop("sum_reward")
    assert abs(sa_r - sb_r) <= 1e-5 * max(1.0, abs(sb_r)), f"{what}: reward sum {sa_r} vs {sb_r}"
    assert ra == rb, f"{what}: statistics differ with final_obs on"


def writes(keep, ids, out, k):
    """The PhysX writes of `_reset_idx` (ART:316-489) for compact reset rows."""
    keep["root_pos_w"][ids] = out.reset_root_state[:k, 0:3]
    keep["root_quat_w"][ids] = out.reset_root_state[:k, 3:7]
    keep["root_lin_vel_w"][ids] = out.reset_root_state[:k, 7:10]
    keep["joint_pos"][ids] = out.reset_joint_pos[:k]
    keep["joint_vel"][ids] = out.reset_joint_vel[:k]
    keep["force_matrix_right"][ids] = 0.0
    keep["force_matrix_left"][ids] = 0.0


def run_fused(N, steps, seed, layout="contiguous", clip=0.0, fall=0.05):
    """Fused steps with final_obs against the oracle and against a twin handle stepped without it."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    sc, orc, origins, (mdp, twin) = setup(N, seed, fall, full_bodies=(layout == "isaac"))
    out = final_buffers(N, obs_clip=clip)
    out_twin = StepBuffers(N, "cuda:0", obs_clip=clip)
    expect = out.final_obs.cpu().clone()
    n_reset = n_time_out = 0
    for step in range(steps):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        _, _, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, None)
        views, keep = to_views(phys, origins, sc.body_indices, layout)
        mdp.step(views, keep["actions"], out)
        twin.step(views, keep["actions"], out_twin)
        torch.cuda.synchronize()
        exact(out.terminated, o_term, f"step {step} terminated")
        exact(out.time_out, o_to, f"step {step} time_out")
        exact(out.dones.nonzero().squeeze(-1), o_ids, f"step {step} reset ids")
        check_final_rows(out, expect, o_ids, expected_final(orc, clip), f"step {step}")
        compare_twins(mdp, twin, out, out_twin, f"step {step}")
        n_reset += len(o_ids)
        n_time_out += int(o_to.sum())
    assert n_reset > 0 and n_time_out > 0


@pytest.mark.parametrize("clip", [0.0, 0.8])
@pytest.mark.parametrize("layout", ["contiguous", "isaac"])
@pytest.mark.parametrize("num_envs", [64, 4096, 1001, (1 << 16) + 44])
def test_fused_step_final_obs_matches_oracle(num_envs, layout, clip):
    """Sizes: one tile, many, a ragged last tile, and the prepared instantiations behind k_prepare*."""
    run_fused(num_envs, 3 if num_envs > 5000 else 5, seed=43 + num_envs, layout=layout, clip=clip,
              fall=0.3 if num_envs == 64 else 0.05)


@pytest.mark.parametrize("device_list", [False, True])
@pytest.mark.parametrize("num_envs,clip", [(1001, 0.0), (4096, 0.8), ((1 << 16) + 44, 0.0)])
def test_three_call_path_final_obs(num_envs, clip, device_list):
    """pass1 / reset / pass2 with host ids or the device-side list: the final rows equal the oracle's and are
    bit-identical to those of a fused step from the same state and inputs (a third handle restored from the 3-call
    handle's snapshot); the other outputs equal a twin without final_obs."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    seed, steps = 43 + num_envs, 4
    sc, orc, origins, (mdp, twin, fused) = setup(num_envs, seed, 0.05, n_mdps=3)
    out = final_buffers(num_envs, obs_clip=clip)
    out_twin = StepBuffers(num_envs, "cuda:0", obs_clip=clip)
    out_fused = final_buffers(num_envs, obs_clip=clip)
    expect = out.final_obs.cpu().clone()
    ep = [orc.episode_length_buf.cuda(), orc.episode_length_buf.cuda()]
    n_reset = 0
    for step in range(steps):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step + 1)  # pass1 advances the Philox step counter before the reset draws
        _, _, _, _, o_ids = orc.step(phys, phys["actions"], m, n, None)
        fused.restore(mdp.snapshot())
        views, keep = to_views(phys, origins, sc.body_indices)
        fused.step(views, keep["actions"], out_fused)
        for h, o, e in ((mdp, out, ep[0]), (twin, out_twin, ep[1])):
            views, keep = to_views(phys, origins, sc.body_indices)
            e += 1
            h.pass1(views, keep["actions"], o, episode_length=e)
            if device_list:
                h.reset(origins, None, o, episode_length=e)
                k = int(o.n_reset.item())
                ids = o.reset_ids[:k].long()
            else:
                ids = o.dones.nonzero().squeeze(-1)
                k = len(ids)
                if k:
                    h.reset(origins, ids, o, episode_length=e)
            if k:
                writes(keep, ids, o, k)
                h.pass2(views, o)
            else:
                h.no_reset()
        torch.cuda.synchronize()
        exact(out.dones.nonzero().squeeze(-1), o_ids, f"step {step} reset ids")
        exact(out_fused.dones.nonzero().squeeze(-1), o_ids, f"step {step} reset ids of the fused step")
        check_final_rows(out, expect, o_ids, expected_final(orc, clip), f"3-call step {step}")
        same_bits(out.final_obs[o_ids], out_fused.final_obs[o_ids],
                  f"3-call step {step}: final_obs differs from the fused step's")
        compare_twins(mdp, twin, out, out_twin, f"3-call step {step}", "device_list" if device_list else "host_ids")
        n_reset += len(o_ids)
    assert n_reset > 0


def test_step_without_reset_leaves_final_obs_untouched():
    """No env resets (the fix-up route of the fused step, as_step_no_reset on the 3-call path): nothing is written."""
    N = 48
    sc, orc, origins, (fused_mdp, three_mdp) = setup(N, 5, 0.0)
    ep = torch.full((N,), 10, dtype=torch.int64)  # (no time-out)
    for m in (fused_mdp, three_mdp):
        m.import_state({"episode_length_buf": ep})
    orc.episode_length_buf[:] = ep
    out_f, out_3 = final_buffers(N), final_buffers(N)
    before = out_f.final_obs.cpu().clone()
    e3 = ep.cuda()
    quiet = 0
    for step in range(4):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        _, _, _, _, o_ids = orc.step(phys, phys["actions"], m, n, None)
        if len(o_ids):
            break  # (the handles would have to reset: the quiet steps before are what this test is about)
        views, keep = to_views(phys, origins, sc.body_indices)
        fused_mdp.step(views, keep["actions"], out_f)
        e3 += 1
        three_mdp.pass1(views, keep["actions"], out_3, episode_length=e3)
        three_mdp.no_reset()
        torch.cuda.synchronize()
        assert not bool(out_f.dones.any()) and not bool(out_3.dones.any())
        same_bits(out_f.final_obs, before, f"step {step}: fused step without a reset wrote final_obs")
        same_bits(out_3.final_obs, before, f"step {step}: pass1 without a reset wrote final_obs")
        quiet += 1
    assert quiet > 0


def test_one_million_envs_final_obs():
    N, seed = 1 << 20, 5
    sc, orc, origins, (mdp,) = setup(N, seed, 0.02, n_mdps=1)
    out = final_buffers(N)
    expect = out.final_obs.cpu().clone()
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    m, n = sc.reset_uniforms(0)
    _, _, o_term, o_to, o_ids = orc.step(phys, phys["actions"], m, n, None)
    views, keep = to_views(phys, origins, sc.body_indices)
    mdp.step(views, keep["actions"], out)
    torch.cuda.synchronize()
    exact(out.dones.nonzero().squeeze(-1), o_ids, "reset ids")
    assert len(o_ids) > 1000
    check_final_rows(out, expect, o_ids, orc.final_obs, "1M envs")


def test_graph_replay_final_obs_equals_eager_steps():
    from allsteps_isaaclab_b200.mdp import PhysicsViews

    N, seed = 4096, 41
    sc, orc, origins, mdps = setup(N, seed, 0.05)
    stones = mdps[0].export_state()["steps_pos"].cpu()
    st = mdps[0].export_state()
    phys = sc.physics(stones, st["curr_target_index"].cpu(), st["swing_leg"].cpu())
    static = {k: v.cuda() for k, v in phys.items()}
    views = PhysicsViews.from_dict(static, origins, sc.body_indices)
    out_g, out_e = final_buffers(N), final_buffers(N)
    graph = mdps[0].capture_step(views, static["actions"], out_g)
    n_reset = 0
    for i in range(5):
        st = mdps[1].export_state()
        phys = sc.physics(st["steps_pos"].cpu(), st["curr_target_index"].cpu(), st["swing_leg"].cpu())
        for k, v in phys.items():
            static[k].copy_(v)
        graph.replay()
        mdps[1].step(views, static["actions"], out_e)
        torch.cuda.synchronize()
        for name in OUTPUTS + ("final_obs",):
            same_bits(getattr(out_g, name), getattr(out_e, name), f"step {i}: {name}")
        n_reset += int(out_e.dones.sum())
    assert n_reset > 0


def test_final_obs_guard_bands_and_determinism():
    """The buffer between guard bands: no kernel writes outside it, fused or 3-call, full or ragged tiles; two runs of
    the same steps give the same bits."""
    from test_gpu_memory_safety import Guarded

    N = 3 * 128 + 44
    results = []
    for run in range(2):
        sc, orc, origins, (mdp,) = setup(N, 61, 0.1, n_mdps=1)
        out = final_buffers(N)
        g = Guarded((N, 59), torch.float32)
        g.t.view(torch.int32).fill_(PREFILL)
        out.final_obs = g.t
        out.step_out.final_obs = g.t.data_ptr()
        ep = orc.episode_length_buf.cuda()
        seen = []
        for step in range(6):
            phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
            views, keep = to_views(phys, origins, sc.body_indices)
            if step % 2 == 0:
                mdp.step(views, keep["actions"], out)
                ep += 1
            else:
                ep += 1
                mdp.pass1(views, keep["actions"], out, episode_length=ep)
                ids = out.dones.nonzero().squeeze(-1)
                if len(ids):
                    mdp.reset(origins, ids, out, episode_length=ep)
                    writes(keep, ids, out, len(ids))
                    mdp.pass2(views, out)
                else:
                    mdp.no_reset()
            torch.cuda.synchronize()
            assert g.intact(), f"run {run} step {step}: a write outside final_obs"
            seen.append(int(out.dones.sum()))
            results.append((run, step, bits(g.t)))
        assert sum(seen) > 0
    for (_, step, a), (_, _, b) in zip(results[:6], results[6:]):
        assert torch.equal(a, b), f"step {step}: final_obs differs between two identical runs"


def test_final_obs_misuse_is_refused():
    from allsteps_isaaclab_b200 import _cabi
    from allsteps_isaaclab_b200.mdp import PhysicsViews, StepBuffers

    N = 256
    sc, orc, origins, (mdp,) = setup(N, 1, 0.05, n_mdps=1)
    phys = {k: v.cuda() for k, v in sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg).items()}
    views = PhysicsViews.from_dict(phys, origins)
    out = StepBuffers(N, "cuda:0")
    spare = torch.zeros(N * 59 + 1, device="cuda")
    base = out.obs.data_ptr()
    for ptr, what in ((base, "final_obs == obs"), (base + 59 * 4 * 100, "overlapping obs"),
                      (base - 59 * 4 * 3, "overlapping the start of obs"), (spare.data_ptr() + 2, "misaligned")):
        out.step_out.final_obs = ptr
        with pytest.raises(_cabi.AllstepsLibraryError, match="final_obs") as e:
            mdp.step(views, phys["actions"], out)
        assert "(-1)" in str(e.value), what
        with pytest.raises(_cabi.AllstepsLibraryError, match="final_obs"):
            mdp.pass1(views, phys["actions"], out)
    out.step_out.final_obs = spare.data_ptr() + 4  # 4-byte aligned, its own memory: accepted
    mdp.step(views, phys["actions"], out)
    torch.cuda.synchronize()


@pytest.mark.parametrize("on", [False, True])
def test_hooks_publish_final_obs(on):
    """StandaloneAllstepsEnv (the DirectRLEnv hook mixin): with the switch on, `extras["final_obs"]` holds the oracle's
    final rows where `reset_buf` is set; with it off there is no such key."""
    from allsteps_isaaclab_b200.env import StandaloneAllstepsEnv
    from test_gpu_faces import _fake_world, _install

    N, seed = 900, 17
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.05)
    st0 = sc.initial_mdp_state()
    st0["episode_length_buf"][::7] = 897
    orc = FinalObsOracle(sc.cfg, N, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    install_mdp_state(orc, st0)
    phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
    robot, left, right = _fake_world(sc, phys)
    scene = types.SimpleNamespace(env_origins=sc.env_origins.cuda())
    env = StandaloneAllstepsEnv(robot, left, right, scene, "cuda:0", sc.cfg, seed=seed, final_obs=on)
    env.mdp.import_state({"steps_pos": orc.steps_pos, "steps_dphi": orc.steps_dphi,
                          **{k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                                 "potentials")}})
    env.episode_length_buf[:] = st0["episode_length_buf"].cuda()
    n_reset = 0
    for step in range(4):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step + 1)
        _, _, _, _, o_ids = orc.step(phys, phys["actions"], m, n, None)
        _install(robot, left, right, phys)
        obs, rew, term, to, extras = env.post_physics_step(phys["actions"].cuda())
        torch.cuda.synchronize()
        exact(env.reset_buf.nonzero().squeeze(-1), o_ids, f"step {step} reset_buf")
        if on:
            fin = extras["final_obs"]
            assert tuple(fin.shape) == (N, 59)
            if len(o_ids):
                close_obs(fin[env.reset_buf], orc.final_obs[o_ids], f"step {step} extras['final_obs']")
        else:
            assert "final_obs" not in extras
        n_reset += len(o_ids)
    assert n_reset > 0
