"""AllstepsCfg -> AsParams (the POD struct the kernels take by value).

Tables the reference builds with torch (`torch.linspace`, ENV:46-47,129) are built with torch here too, so their
fp32 values are identical to the reference's.
"""
from __future__ import annotations

import numbers

import torch

from . import _cabi
from .config import AllstepsCfg, NUM_JOINTS


def _f32(x: float) -> float:
    return float(torch.tensor(x, dtype=torch.float64).to(torch.float32))


def make_params(cfg: AllstepsCfg, seed: int = 0, flags: int = 0, grid_bins: int = 0,
                joint_limits=None) -> _cabi.AsParams:
    """joint_limits: optional (J,2) tensor / nested list [lower, upper] in radians, as the simulator reports them
    (`robot.data.joint_pos_limits[0]`); default: the MJCF ranges converted in double (config.py)."""
    S = cfg.num_steps
    if isinstance(S, bool) or not isinstance(S, numbers.Integral) or not _cabi.MIN_STONES <= S <= _cabi.MAX_STONES:
        raise ValueError(f"num_steps must be an integer in {_cabi.MIN_STONES}..{_cabi.MAX_STONES} (CFG:90), got {S!r}")
    p = _cabi.AsParams()
    p.num_steps = int(S)
    n_levels = cfg.max_curriculum + 1
    assert n_levels <= _cabi.NUM_LEVELS
    p.step_dt = cfg.step_dt
    p.max_episode_length = cfg.max_episode_length
    p.step_radius = cfg.step_radius
    p.dist_lower = cfg.dist_range[0]
    dist_lohi = torch.tensor(cfg.dist_range, dtype=torch.float32)
    dist_upper = torch.linspace(*dist_lohi, n_levels)  # ENV:129
    term_h = torch.linspace(*cfg.termination_height_range, n_levels)  # ENV:46
    gain = torch.linspace(*cfg.applied_gain_range, n_levels)  # ENV:47
    for i in range(_cabi.NUM_LEVELS):
        k = min(i, n_levels - 1)
        p.dist_upper[i] = float(dist_upper[k])
        p.termination_height[i] = float(term_h[k])
        p.applied_gain[i] = float(gain[k])
    p.yaw_range_deg[0], p.yaw_range_deg[1] = cfg.yaw_range_deg
    p.pitch_range_deg[0], p.pitch_range_deg[1] = cfg.pitch_range_deg
    p.init_step_separation = cfg.init_step_separation
    p.max_level = cfg.max_curriculum
    p.progress_threshold = cfg.curriculum_progress_threshold
    p.contact_epsilon = cfg.contact_epsilon
    p.stop_frames = cfg.stop_frames
    p.energy_cost_scale = cfg.energy_cost_scale
    p.actions_cost_scale = cfg.actions_cost_scale
    p.alive_reward_scale = cfg.alive_reward_scale
    p.dof_vel_scale = cfg.dof_vel_scale
    p.joint_at_limit_cost_scale = cfg.joint_at_limit_cost_scale
    p.death_cost = cfg.death_cost
    p.termination_height_absolute = cfg.termination_height_absolute
    p.max_root_speed = cfg.max_root_speed
    p.missed_step_height = cfg.missed_step_height
    lo, hi = cfg.initial_joint_angle_range
    p.noise_span = hi - lo  # MATH:1331 evaluates (upper - lower) in Python double, then rounds to fp32
    p.noise_lower = lo
    p.clip_lower, p.clip_upper = cfg.initial_joint_angle_clip_range
    for i in range(3):
        p.default_root_pos[i] = cfg.default_root_pos[i]
    limits = cfg.joint_limits_rad()
    if joint_limits is not None:
        jl = torch.as_tensor(joint_limits, dtype=torch.float32).cpu()
        if tuple(jl.shape) != (NUM_JOINTS, 2):
            raise ValueError(f"joint_limits must be ({NUM_JOINTS},2), got {tuple(jl.shape)}")
        limits = [(float(a), float(b)) for a, b in jl.tolist()]
    pose = cfg.reset_joint_pose()
    src, sign = cfg.mirror_permutation()
    for j in range(NUM_JOINTS):
        p.joint_lower[j] = limits[j][0]
        p.joint_upper[j] = limits[j][1]
        p.joint_gears[j] = cfg.joint_gears[j]
        p.reset_pose[j] = pose[j]
        p.mirror_src[j] = src[j]
        p.mirror_sign[j] = sign[j]
    p.flags = flags
    p.grid_bins = grid_bins
    p.seed = seed
    return p
