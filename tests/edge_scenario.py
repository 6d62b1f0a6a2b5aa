"""A one-step scenario whose decisions sit on their thresholds, with operands both sides compute exactly (test data).

Every env starts from one quiet pose: stones on the x axis 0.75 m apart with the current stone at the env's origin,
root over the previous stone at 1.3 m, identity orientation, no velocity, joints at mid-range, feet on the ground
(z = 0) with the swing foot 1 m past the stone, no contact, no action.  Each edge env then changes one quantity so
that one comparison of ENV:396-457 / ENV:350-375 is decided by it, at `nextafter(threshold, -inf)`, at the threshold
and at `nextafter(threshold, +inf)`:

    speed                 |v| = |v_x|                        vs 1.6 (speed cost) and max_root_speed (so_fast)
    root z                                                   vs termination_height_absolute (died)
    h                     torso z - 0                        vs termination_height[level], every level (fell)
    contact norm          |f_z| on the current stone column  vs contact_epsilon (pressed), right and left foot
    foot distance         |x_foot - 0|                       vs step_radius, swing leg and stance leg
    |scaled joint|        positions found by bisection       vs 0.99 (joint-at-limit cost)
    episode length        897 / 898 / 899 before the increment (time_out)
    actions               +-1 and one ulp beyond, 1.5, 0.5   clamp -> action and energy cost (joint velocities 1:
                                                             sums of 21 equal terms, exact in any order)
    idx                   18 / 19 with the count reaching 1 or 2: the step reward is paid below S-1 only; 19 clamps
    body distance         |0 - (-d)| at idx 19               vs 0.15 (target bonus)

Norms of axis-aligned vectors are exact (sqrt(x*x) == |x| in IEEE arithmetic); so are the differences with zero.  So
every mask, and every term but the progress, step reward and the two angles, is exact on both sides: a mismatch is a
bug, not noise.  atan2 is not bit-exact between the two sides, so roll and pitch are placed 1e-4 rad around 0.4 and at
tiny negative angles (-1e-3, -1e-6 rad), which wrap to just under 2*pi and pay a ~6.28 cost.
"""
from __future__ import annotations

import math
from typing import Dict, List, Tuple

import numpy as np
import torch

from allsteps_isaaclab_b200 import synthetic as syn
from allsteps_isaaclab_b200.config import AllstepsCfg, NUM_JOINTS, NUM_STONES
from oracle import allsteps_oracle as ao

BASE_IDX = 5
ROOT_Z = 1.3
TORSO_Z = 1.55
# reward-term columns that are exact on every edge env (alive, speed, energy, action, joint-at-limit, bonus)
EXACT_TERM_COLUMNS = (0, 4, 5, 6, 7, 9)


def f32(x) -> np.float32:
    return np.float32(x)


def below(x) -> float:
    return float(np.nextafter(f32(x), f32(-np.inf)))


def above(x) -> float:
    return float(np.nextafter(f32(x), f32(np.inf)))


def around(x) -> Tuple[float, float, float]:
    x = float(f32(x))
    return below(x), x, above(x)


def limit_crossings(cfg: AllstepsCfg) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per joint, the fp32 positions whose `scale_to_unit` (the oracle's, in fp32) is the last one not beyond the
    limit cost's 0.99 on the upper side (largest x with scaled <= 0.99) and on the lower side (smallest x with
    scaled >= -0.99).  Found by bisection over the ordered fp32 bit patterns of the joint's range."""
    lim = syn.joint_limits_tensor(cfg)
    lo, hi = lim[:, 0], lim[:, 1]

    def scaled(bits: torch.Tensor) -> torch.Tensor:
        return ao.scale_to_unit(ordered_to_float(bits), lo, hi)

    mid = float_to_ordered((lo + hi) * 0.5)
    far_hi = float_to_ordered(hi + (hi - lo))
    far_lo = float_to_ordered(lo - (hi - lo))
    # upper: largest x with scaled(x) <= 0.99 in [mid, far_hi]
    a, b = mid.clone(), far_hi.clone()
    while bool((b - a > 1).any()):
        m = (a + b) // 2
        ok = scaled(m) <= 0.99
        a = torch.where(ok, m, a)
        b = torch.where(ok, b, m)
    upper = ordered_to_float(a)
    # lower: smallest x with scaled(x) >= -0.99 in [far_lo, mid]
    a, b = far_lo.clone(), mid.clone()
    while bool((b - a > 1).any()):
        m = (a + b) // 2
        ok = scaled(m) >= -0.99
        b = torch.where(ok, m, b)
        a = torch.where(ok, a, m)
    lower = ordered_to_float(b)
    return lower, upper


def float_to_ordered(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> int64 keys whose order is the order of the floats (one step = one ulp)."""
    i = x.to(torch.float32).view(torch.int32).to(torch.int64)
    return torch.where(i < 0, -(i & 0x7FFFFFFF), i)


def ordered_to_float(k: torch.Tensor) -> torch.Tensor:
    i = torch.where(k < 0, (-k) | (-0x80000000), k)
    return i.to(torch.int32).view(torch.float32)


class EdgeScenario:
    """`self.groups[name]` are the env rows of one boundary (three per boundary, in the order -1 ulp / at / +1 ulp
    unless stated); `copies` places the edge envs again at every given row offset, the rows in between are quiet envs."""

    def __init__(self, copies: Tuple[int, ...] = (0,), num_envs: int = 0, seed: int = 5):
        self.cfg = cfg = AllstepsCfg()
        self.seed = seed
        S, J = NUM_STONES, NUM_JOINTS
        lim = syn.joint_limits_tensor(cfg)
        self.joint_limits = lim
        mid = (lim[:, 0] + lim[:, 1]) * 0.5
        term_h = torch.linspace(*cfg.termination_height_range, cfg.max_curriculum + 1)
        specs: List[Dict] = []
        self.groups: Dict[str, List[int]] = {}

        def add(group, **kw):
            self.groups.setdefault(group, []).append(len(specs))
            specs.append(kw)

        for s in around(1.6):
            add("speed_cost", v=s)
        for s in around(cfg.max_root_speed):
            add("so_fast", v=s)
        for z in around(cfg.termination_height_absolute):
            add("died", root_z=z)
        for level in range(cfg.max_curriculum + 1):
            for z in around(float(term_h[level])):
                add(f"fell_level{level}", level=level, torso_z=z)
        for c in around(cfg.contact_epsilon):
            add("pressed_right_swing", leg=0, right=(0.0, 0.0), f_right=c)
        for c in around(cfg.contact_epsilon):
            add("pressed_left_swing", leg=1, left=(0.0, 0.0), right=(-0.75, 0.0), f_left=c)
        for c in around(cfg.contact_epsilon):
            add("pressed_left_stance", leg=0, left=(0.0, 0.0), f_left=c)
        for d in around(cfg.step_radius):
            add("radius_right_swing", leg=0, right=(d, 0.0), f_right=100.0)
        for d in around(cfg.step_radius):
            add("radius_left_swing", leg=1, left=(d, 0.0), right=(-0.75, 0.0), f_left=100.0)
        for d in around(cfg.step_radius):
            add("radius_left_stance", leg=0, left=(d, 0.0), f_left=100.0, f_right=100.0)
        lower, upper = limit_crossings(cfg)
        up = torch.stack([torch.nextafter(upper, torch.full_like(upper, -math.inf)), upper,
                          torch.nextafter(upper, torch.full_like(upper, math.inf))])
        dn = torch.stack([torch.nextafter(lower, torch.full_like(lower, -math.inf)), lower,
                          torch.nextafter(lower, torch.full_like(lower, math.inf))])
        for k in range(3):
            add("joint_limit_upper", joints=up[k])
        for k in range(3):
            add("joint_limit_lower", joints=dn[k])
        for ep in (897, 898, 899):
            add("time_out", ep=ep)
        for a in (0.5, 1.0, above(1.0), 1.5, -1.0, below(-1.0)):
            add("action_clamp", act=a)
        # reached in pass 1 (swing foot on the stone, pressed) with the count going to 1 (pays below S-1 only) or to 2
        # (advances; at S-1 the index clamps)
        for idx, count in ((18, 0), (19, 0), (18, 1), (19, 1)):
            add("last_stones", idx=idx, count=count, right=(0.0, 0.0), f_right=100.0)
        for d in around(0.15):
            add("target_bonus", idx=S - 1, root_x=-d)
        for theta in (0.4 - 1e-4, 0.4 + 1e-4, -1e-3, -1e-6):
            add("roll", roll=theta)
        for theta in (0.4 - 1e-4, 0.4 + 1e-4, -1e-3, -1e-6):
            add("pitch", pitch=theta)
        self.num_edge = E = len(specs)

        N = num_envs or (max(copies) + E)
        assert all(o + E <= N for o in copies)
        self.N = N
        self.edge_rows = torch.cat([torch.arange(E) + o for o in copies])
        self.body_indices = (0, 1, 2)
        self.env_origins = torch.zeros(N, 3)
        idx = torch.full((N,), BASE_IDX, dtype=torch.int64)
        leg = torch.zeros(N, dtype=torch.int64)
        count = torch.zeros(N, dtype=torch.int64)
        ep = torch.full((N,), 100, dtype=torch.int64)
        level = torch.zeros(N, dtype=torch.int64)
        root = torch.tensor([-0.75, 0.0, ROOT_Z]).repeat(N, 1)
        quat = torch.tensor([1.0, 0.0, 0.0, 0.0]).repeat(N, 1)
        vel = torch.zeros(N, 3)
        body = torch.zeros(N, 3, 3)
        body[:, 0] = torch.tensor([1.0, 0.0, 0.0])    # right foot: the swing foot, 1 m past its stone
        body[:, 1] = torch.tensor([-0.75, 0.0, 0.0])  # left foot: on the previous stone
        body[:, 2] = torch.tensor([-0.75, 0.0, TORSO_Z])
        joint_pos = mid.repeat(N, 1)
        joint_vel = torch.zeros(N, J)
        actions = torch.zeros(N, J)
        f_right = torch.zeros(N, 1, S, 3)
        f_left = torch.zeros(N, 1, S, 3)
        for o in copies:
            for i, kw in enumerate(specs):
                e = o + i
                idx[e] = kw.get("idx", BASE_IDX)
                leg[e] = kw.get("leg", 0)
                count[e] = kw.get("count", 0)
                ep[e] = kw.get("ep", 100)
                level[e] = kw.get("level", 0)
                if "v" in kw:
                    vel[e, 0] = kw["v"]
                if "root_z" in kw:
                    root[e, 2] = kw["root_z"]
                if "root_x" in kw:
                    root[e, 0] = kw["root_x"]
                if "torso_z" in kw:
                    body[e, 2, 2] = kw["torso_z"]
                if "right" in kw:
                    body[e, 0, 0:2] = torch.tensor(kw["right"])
                if "left" in kw:
                    body[e, 1, 0:2] = torch.tensor(kw["left"])
                if "f_right" in kw:
                    f_right[e, 0, idx[e], 2] = kw["f_right"]
                if "f_left" in kw:
                    f_left[e, 0, idx[e], 2] = kw["f_left"]
                if "joints" in kw:
                    joint_pos[e] = kw["joints"]
                if "act" in kw:
                    actions[e] = kw["act"]
                    joint_vel[e] = 1.0
                if "roll" in kw:
                    h = kw["roll"] / 2
                    quat[e] = torch.tensor([math.cos(h), math.sin(h), 0.0, 0.0])
                if "pitch" in kw:
                    h = kw["pitch"] / 2
                    quat[e] = torch.tensor([math.cos(h), 0.0, math.sin(h), 0.0])
        # stones on the x axis, 0.75 m apart, the current one at the origin
        k = torch.arange(S, dtype=torch.float32)
        self.steps_pos = torch.zeros(N, S, 3)
        self.steps_pos[:, :, 0] = (k[None, :] - idx[:, None].float()) * 0.75
        self.steps_dphi = torch.zeros(N, S)
        self.state = {"curr_target_index": idx, "swing_leg": leg, "target_reach_count": count,
                      "episode_length_buf": ep, "curriculum": level, "potentials": torch.full((N,), -60.0)}
        self.phys = {"root_pos_w": root, "root_quat_w": quat, "root_lin_vel_w": vel, "root_ang_vel_w": torch.zeros(N, 3),
                     "body_pos_w": body, "joint_pos": joint_pos, "joint_vel": joint_vel,
                     "force_matrix_right": f_right, "force_matrix_left": f_left, "actions": actions}

    def rows(self, group: str) -> torch.Tensor:
        """Rows of `group` in every copy."""
        base = torch.tensor(self.groups[group])
        offs = self.edge_rows[:: self.num_edge] if self.num_edge else torch.zeros(0, dtype=torch.int64)
        return torch.cat([base + int(o) for o in offs])

    def install(self, orc):
        """Put the scenario's MDP state and stones into an oracle."""
        for name in ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "curriculum"):
            getattr(orc, name)[:] = self.state[name]
        orc.potentials = self.state["potentials"].clone()
        orc.old_potentials = self.state["potentials"].clone()
        orc.prev_target_index = torch.clamp(orc.curr_target_index - 1, 0, NUM_STONES - 1)
        orc.next_target_index = torch.clamp(orc.curr_target_index + 1, 0, NUM_STONES - 1)
        orc.steps_pos[:] = self.steps_pos
        orc.steps_dphi[:] = self.steps_dphi

    def reset_uniforms(self, step: int):
        from oracle import philox

        m, n = philox.reset_tables(self.seed, step, np.arange(self.N, dtype=np.int64))
        return torch.from_numpy(m), torch.from_numpy(n)


def branch_outcomes(sc: EdgeScenario, orc) -> Dict[str, Tuple[torch.Tensor, torch.Tensor]]:
    """Per boundary: (rows, decision) after one oracle step of the scenario -- the mask whose threshold the rows
    straddle, evaluated on the oracle's pass-1 state (`TermsOracle` terms and masks)."""
    t = orc.terms
    out = {}

    def put(name, group, decision):
        r = sc.rows(group)
        out[name] = (r, decision[r])

    put("speed_cost", "speed_cost", t[:, 4] > 0)
    put("so_fast", "so_fast", orc.so_fast)
    put("died", "died", orc.died)
    for level in range(sc.cfg.max_curriculum + 1):
        put(f"fell_level{level}", f"fell_level{level}", orc.fell)
    contacts = orc.pass1_foot_contact
    put("pressed_right_swing", "pressed_right_swing", contacts[:, 0] > 0)
    put("pressed_left_swing", "pressed_left_swing", contacts[:, 1] > 0)
    put("pressed_left_stance", "pressed_left_stance", contacts[:, 1] > 0)
    put("radius_right_swing", "radius_right_swing", orc.pass1_target_reached)
    put("radius_left_swing", "radius_left_swing", orc.pass1_target_reached)
    put("radius_left_stance", "radius_left_stance", orc.pass1_foot_dist[:, 1] < sc.cfg.step_radius)
    limit_any = (orc.joint_pos_scaled_pass1.abs() > 0.99).any(-1)
    put("joint_limit_upper", "joint_limit_upper", limit_any)
    put("joint_limit_lower", "joint_limit_lower", limit_any)
    put("time_out", "time_out", orc.reset_time_outs)
    put("action_clamp", "action_clamp", orc.actions.abs().amax(-1) < sc.phys["actions"].abs().amax(-1))
    put("step_reward", "last_stones", t[:, 8] > 0)
    put("advance", "last_stones", orc.advanced1)
    put("target_bonus", "target_bonus", t[:, 9] > 0)
    put("roll_cost", "roll", t[:, 2] > 0)
    put("pitch_cost", "pitch", t[:, 3] > 0)
    return out
