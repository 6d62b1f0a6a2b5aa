"""CPU checks of the step-variant parity suite: the recording oracle stays the pinned port, the case table of
tests/test_gpu_step_variants.py names every `k_step` instantiation, and the edge scenario straddles every boundary."""
from __future__ import annotations

import pytest
import torch

import edge_scenario as edge
import step_variants as sv
from scenario import Scenario, install_mdp_state
from terms_oracle import STAT_FIELDS, TermsOracle, signed_total


@pytest.mark.parametrize("num_envs,seed,high_index", [(512, 11, False), (2048, 13, True), (300, 61, False)])
def test_recorded_terms_add_up_to_the_oracle_reward_bit_for_bit(num_envs, seed, high_index):
    sc = Scenario(num_envs, seed=seed, fall_fraction=0.05)
    st0 = sc.initial_mdp_state(per_env_levels=True)
    if high_index:
        st0["curr_target_index"] = torch.randint(15, 20, (num_envs,), generator=sc.gen)
    orc = TermsOracle(sc.cfg, num_envs, sc.env_origins, sc.joint_limits, sc.body_indices, sc.stone_uniforms(0))
    install_mdp_state(orc, st0)
    orc.curriculum[:] = st0["curriculum"]
    seen = torch.zeros(10, dtype=torch.bool)
    for step in range(4):
        phys = sc.physics(orc.steps_pos, orc.curr_target_index, orc.swing_leg)
        m, n = sc.reset_uniforms(step)
        _, reward, term, time_out, ids = orc.step(phys, phys["actions"], m, n, None)
        t = orc.terms
        assert t.shape == (num_envs, 10) and t.dtype == torch.float32
        alive = ~term
        assert torch.equal(signed_total(t)[alive], reward[alive]), f"step {step}: terms do not add up to the reward"
        assert bool((reward[term] == sc.cfg.death_cost).all())
        assert bool((t[:, 2:8] >= 0).all()), "costs are recorded positive"
        seen |= (t != 0).any(0)
        s = orc.stats
        assert set(s) == set(STAT_FIELDS)
        assert s["n_reset"] == len(ids) == int((term | time_out).sum())
        assert s["n_terminated"] <= s["n_fell"] + s["n_so_fast"] + s["n_died"]
        assert s["step_counter"] == step
        assert s["n_advanced"] >= int(orc.advanced1.sum())
        assert abs(orc.reward_sum - float(reward.double().sum())) == 0.0
    # (the target bonus almost never fires in the synthetic scenarios; the edge scenario places it)
    assert bool(seen[:9].all()), f"terms never nonzero: {(~seen).nonzero().flatten().tolist()}"


def test_case_table_names_every_step_kernel_instantiation():
    variants = sv.parse_step_variants()
    assert len(variants) == 18, f"kStepVariants has {len(variants)} rows"
    assert len({v.template for v in variants}) == len(variants), "two rows with one instantiation"
    by_row = sv.rows_by_number(variants)
    named = {r for c in sv.CASES for r in c.rows}
    missing = sorted(set(by_row) - named)
    assert not missing, f"kStepVariants rows without a case in tests/step_variants.py: {missing}"
    assert named <= set(by_row), f"cases name rows kStepVariants does not have: {sorted(named - set(by_row))}"
    assert len({c.name for c in sv.CASES}) == len(sv.CASES)


@pytest.mark.parametrize("case", sv.CASES, ids=lambda c: c.name)
def test_case_rows_follow_from_the_case_conditions(case):
    """The rows a case claims agree with its conditions: mode, ragged tail, prepared / two-FMA / run-time division,
    FAST and PACKED (the triggers of the generic instantiation)."""
    by_row = sv.rows_by_number(sv.parse_step_variants())
    full, *rest = [by_row[r] for r in case.rows]
    assert all(v.mode == case.mode for v in (full, *rest))
    ragged = case.num_envs % sv.TILE != 0
    assert [v.kind for v in rest] == (["ragged"] if ragged else [])
    if case.mode == "pass2" or case.exact_div or (case.mode == "pass1" and not case.prepared):
        kind = "runtime-div"
    else:
        kind = "prepared" if case.prepared else "two-fma"
    assert full.kind == kind
    variants = kind in ("prepared", "two-fma")
    assert full.fast == (variants and case.fast)
    assert full.packed == (variants and case.packed)
    assert full.template[2] and all(not v.template[2] for v in rest)  # FULL


def test_case_table_covers_every_generic_trigger():
    triggers = {o for c in sv.CASES if c.mode != "pass2" for o in c.outputs}
    assert triggers == {"reward_terms", "obs_clip", "final_obs", "quat_xyzw"}


def test_kernel_names_parse():
    name = "void as::k_step<2, 0, true, true, false, true>(as::StepArgs)"
    assert sv.parse_kernel_name(name) == (2, 0, True, True, False, True)
    assert sv.parse_kernel_name("void as::k_fixup_finish(as::StepArgs)") is None


# the fewest envs on each side of a boundary (per copy of the scenario)
MIN_HITS = {"so_fast": (1, 2), "died": (1, 2), "speed_cost": (1, 2), "time_out": (2, 1), "action_clamp": (3, 3),
            "step_reward": (1, 3), "advance": (2, 2), "target_bonus": (1, 2), "roll_cost": (3, 1),
            "pitch_cost": (3, 1), "joint_limit_upper": (1, 2), "joint_limit_lower": (1, 2),
            "radius_right_swing": (1, 2), "radius_left_swing": (1, 2), "radius_left_stance": (1, 2),
            "pressed_right_swing": (1, 2), "pressed_left_swing": (1, 2), "pressed_left_stance": (1, 2),
            **{f"fell_level{k}": (1, 2) for k in range(10)}}


def run_edge_oracle(sc):
    orc = TermsOracle(sc.cfg, sc.N, sc.env_origins, sc.joint_limits, sc.body_indices, None)
    sc.install(orc)
    m, n = sc.reset_uniforms(0)
    orc.step(sc.phys, sc.phys["actions"], m, n, None)
    return orc


def test_edge_scenario_lands_on_both_sides_of_every_boundary():
    sc = edge.EdgeScenario(copies=(0, 256))
    orc = run_edge_oracle(sc)
    outcomes = edge.branch_outcomes(sc, orc)
    assert set(outcomes) == set(MIN_HITS)
    for name, (rows, decision) in outcomes.items():
        yes, no = int(decision.sum()) // 2, int((~decision).sum()) // 2
        want_yes, want_no = MIN_HITS[name]
        assert yes >= want_yes and no >= want_no, f"{name}: taken {yes}, not taken {no} per copy; want {MIN_HITS[name]}"
    # the branch flips between the last two edge values (+1 ulp) for the threshold groups: the threshold itself
    # decides the same way as -1 ulp for the strict comparisons
    for name in ("speed_cost", "so_fast", "pressed_right_swing", "pressed_left_swing", "pressed_left_stance",
                 "joint_limit_upper"):
        rows, decision = outcomes[name]
        assert decision[:3].tolist() == [False, False, True], name
    for name in ("died", "radius_right_swing", "radius_left_swing", "radius_left_stance", "target_bonus",
                 "joint_limit_lower", *(f"fell_level{k}" for k in range(10))):
        rows, decision = outcomes[name]
        assert decision[:3].tolist() == [True, False, False], name
    assert outcomes["time_out"][1][:3].tolist() == [False, True, True]


def test_edge_scenario_operands_are_exact():
    """The operands of the decisions are the values placed: an exact norm, an exact difference."""
    sc = edge.EdgeScenario()
    orc = run_edge_oracle(sc)
    r = sc.rows("speed_cost")
    assert torch.equal(orc.terms[r, 4], torch.tensor([0.0, 0.0, edge.above(1.6) - edge.f32(1.6)]))
    r = sc.rows("target_bonus")
    assert torch.equal(orc.body_dist_to_target_xy[r], torch.tensor(edge.around(0.15)))
    for level in range(10):
        r = sc.rows(f"fell_level{level}")
        assert torch.equal(orc.torso_to_feet_height[r], sc.phys["body_pos_w"][r, 2, 2])
    r = sc.rows("radius_right_swing")
    assert torch.equal(orc.pass1_foot_dist[r, 0], torch.tensor(edge.around(0.25)))
    r = sc.rows("action_clamp")
    energy = torch.tensor([10.5, 21.0, 21.0, 21.0, 21.0, 21.0]) * edge.f32(0.009)
    assert torch.equal(orc.terms[r, 5], energy)
    # the pre-step stones of the edge envs are the hand-placed ones, so nothing about them was drawn
    assert orc.stats["n_reset"] > 0 and orc.stats["n_regenerated"] == 0
