"""B2 face: Isaac Lab manager terms `func(env, **params) -> torch.Tensor` for the Allsteps task.

The reference task is a `DirectRLEnv` (SURVEY D1); `BASELINE.json:north_star` also asks for the manager-term surface
(ObservationManager / RewardManager / TerminationManager / EventManager reset / CurriculumManager).  These functions
satisfy the call conventions of the reference's managers:

    observation  f(env, **params) -> (N, d)      observation_manager.py:308   (cat order = cfg order => 59 columns)
    reward       f(env, **params) -> (N,)        reward_manager.py:148        (manager multiplies by weight * dt)
    termination  f(env, **params) -> (N,) bool   termination_manager.py:165
    event reset  f(env, env_ids, **params)       event_manager.py:240
    curriculum   f(env, env_ids, **params)       curriculum_manager.py:138

All terms of one env step are slices of ONE kernel launch: the first term that needs results runs pass 1 (cached on
`env.common_step_counter`), `reset_allsteps` runs the masked reset + pass 2, observation terms slice the observation
buffer.  `env` needs: `num_envs`, `device`, `common_step_counter`, `episode_length_buf`, `scene` holding
`env_origins` and the entities named by the params (`scene["robot"]`, `scene["foot_contacts_left/right"]`), and
`action_manager.action` (or `env.actions`).

No term steps the MDP before the first env step: `ObservationManager._prepare_terms` calls every observation term
once AT CONSTRUCTION to read its shape (observation_manager.py:411), and `ManagerBasedRLEnv.reset()` computes
observations after the reset events with `common_step_counter == 0`; in both cases the terms hand out the buffers as
they are (zeros, or what `reset_allsteps` left there) and launch nothing.  Every term takes the optional parameters
`asset_cfg` / `left_sensor_cfg` / `right_sensor_cfg` (a `SceneEntityCfg` or a name) to name its scene entities, the
way Isaac Lab's stock terms do; `manager_cfg.py` assembles the term configurations the managers take.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .config import AllstepsCfg
from .mdp import AllstepsMDP, PhysicsViews, StepBuffers

_KEY = "_allsteps_b200"

# observation columns, ENV:330-343
OBS_SLICES = {"torso_to_feet_height": (0, 1), "root_roll_pitch": (1, 3), "root_lin_vel_b": (3, 6),
              "joint_pos_scaled": (6, 27), "joint_vel_scaled_clipped": (27, 48), "foot_contact": (48, 50),
              "stone_targets_b": (50, 59)}
# AsStepOut.reward_terms columns (costs are positive numbers)
REWARD_COLUMNS = {"alive": 0, "progress": 1, "roll_cost": 2, "pitch_cost": 3, "speed_cost": 4, "energy_cost": 5,
                  "action_cost": 6, "joint_at_limit_cost": 7, "step_reward": 8, "target_bonus": 9}
DEFAULT_ENTITIES = ("robot", "foot_contacts_left", "foot_contacts_right")


def _entity_name(cfg, default: str) -> str:
    """A `SceneEntityCfg` (manager_base.py:250-266 resolves it against env.scene), a plain name, or None."""
    if cfg is None:
        return default
    return cfg if isinstance(cfg, str) else cfg.name


class _Binding:
    """Per-env glue shared by all terms: the MDP object, the output buffers and the per-step cache."""

    def __init__(self, env, robot="robot", left="foot_contacts_left", right="foot_contacts_right", seed=0,
                 task_cfg: Optional[AllstepsCfg] = None, grid_bins: int = 0, intended_regen: bool = False,
                 distributed: bool = False):
        """grid_bins / intended_regen: the `AllstepsMDP` extensions (difficulty-grid curriculum with grid_bins per
        axis; regeneration of the stones of envs that had passed half of them).  Both regenerate stones in
        `reset_allsteps`, which then writes them to the scene's stone collection.  distributed: this env is one
        rank's shard of a torchrun job -- global env ids after the other ranks' and the global 3-call mode (see
        `AllstepsHooksB200._init_allsteps_b200`)."""
        from .env import resolve_robot_tables

        self.cfg = task_cfg or AllstepsCfg()
        self.names = (robot, left, right)
        dev = torch.device(env.device)
        self.body_rows, joint_limits = resolve_robot_tables(env.scene[robot], self.cfg)
        offset = 0
        if distributed:
            from .sharding import global_env_offset

            offset = global_env_offset(env.num_envs, dev)
        self.mdp = AllstepsMDP(env.num_envs, device=dev, cfg=self.cfg, seed=seed, joint_limits=joint_limits,
                               grid_bins=grid_bins, intended_regen=intended_regen, env_id_offset=offset)
        if distributed:
            self.mdp.connect_peers(three_call=True)
        self.buf = StepBuffers(env.num_envs, dev, reward_terms=True)
        self.buf.obs.zero_()
        self.buf.reward.zero_()
        self.buf.reward_terms.zero_()
        self.mdp.generate_stones(env.scene.env_origins)
        self.epoch = None
        self.open = False

    def views(self, env) -> PhysicsViews:
        robot, left, right = (env.scene[n] for n in self.names)
        d = robot.data
        t = (d.root_pos_w, d.root_quat_w, d.root_lin_vel_w, d.body_pos_w, d.joint_pos, d.joint_vel,
             right.data.force_matrix_w, left.data.force_matrix_w, env.scene.env_origins)
        return PhysicsViews.cached(self, t, self.body_rows)

    def ensure_pass1(self, env):
        """Pass 1 of the env step in progress, once.  Before the first step (`common_step_counter == 0`: the shape
        probe at manager construction, the observations of the initial `reset()`) nothing is launched."""
        if env.common_step_counter == 0 or self.epoch == env.common_step_counter:
            return
        am = getattr(env, "action_manager", None)
        actions = am.action if am is not None else env.actions
        self.mdp.pass1(self.views(env), actions, self.buf, episode_length=env.episode_length_buf)
        self.epoch = env.common_step_counter
        self.open = True  # closed by `reset_allsteps` (pass 2) or by the first observation term when nothing resets


def binding(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None, **kw) -> _Binding:
    b = getattr(env, _KEY, None)
    if b is None:
        names = (_entity_name(asset_cfg, DEFAULT_ENTITIES[0]), _entity_name(left_sensor_cfg, DEFAULT_ENTITIES[1]),
                 _entity_name(right_sensor_cfg, DEFAULT_ENTITIES[2]))
        b = _Binding(env, *names, **kw)
        setattr(env, _KEY, b)
    return b


# ---------------------------------------------------------------------------------------------- observations
def _obs(env, name: str, ent) -> torch.Tensor:
    b = binding(env, *ent)
    b.ensure_pass1(env)  # no-op when termination/reward terms already ran this step (the usual order)
    if b.open:  # observations are computed after `_reset_idx` (manager_based_rl_env.py:220-239): nothing reset this step
        b.mdp.no_reset()
        b.open = False
    lo, hi = OBS_SLICES[name]
    return b.buf.obs[:, lo:hi]


def torso_to_feet_height(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:332
    return _obs(env, "torso_to_feet_height", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


def root_roll_pitch(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:333-334
    return _obs(env, "root_roll_pitch", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


def root_lin_vel_b(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:335
    return _obs(env, "root_lin_vel_b", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


def joint_pos_scaled(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:336
    return _obs(env, "joint_pos_scaled", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


def joint_vel_scaled_clipped(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:337
    return _obs(env, "joint_vel_scaled_clipped", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


def foot_contact(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:338
    return _obs(env, "foot_contact", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


def stone_targets_b(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:  # ENV:339
    return _obs(env, "stone_targets_b", (asset_cfg, left_sensor_cfg, right_sensor_cfg))


OBSERVATION_TERMS = (torso_to_feet_height, root_roll_pitch, root_lin_vel_b, joint_pos_scaled,
                     joint_vel_scaled_clipped, foot_contact, stone_targets_b)


# ---------------------------------------------------------------------------------------------- rewards
def allsteps_total_reward(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:
    """ENV:377-394 in one term.  RewardManager multiplies by `weight * dt` (reward_manager.py:148): use
    weight = 1 / env.step_dt to reproduce the DirectRLEnv reward (to within the two roundings of `x * w * dt`)."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    b.ensure_pass1(env)
    return b.buf.reward


def reward_term(env, name: str, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:
    """One of the ten terms of ENV:350-375 (see REWARD_COLUMNS; costs are returned positive, give them a negative
    weight).  Their signed sum equals `allsteps_total_reward` for envs that did not terminate."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    b.ensure_pass1(env)
    return b.buf.reward_terms[:, REWARD_COLUMNS[name]]


# ---------------------------------------------------------------------------------------------- terminations
def allsteps_terminated(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:
    """ENV:401-405 fell | so_fast | died."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    b.ensure_pass1(env)
    return b.buf.terminated


def allsteps_time_out(env, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> torch.Tensor:
    """ENV:399: `episode_length_buf >= max_episode_length - 1` (the stock mdp.time_out uses `>= max`)."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    b.ensure_pass1(env)
    return b.buf.time_out


# ---------------------------------------------------------------------------------------------- reset event
def reset_allsteps(env, env_ids, write_to_sim: bool = True, asset_cfg=None, left_sensor_cfg=None,
                   right_sensor_cfg=None, stones_cfg="steps"):
    """EventManager `mode="reset"` term, ENV:469-567: MDP reset + start pose + PhysX writes + pass 2.  `env_ids` is
    what EventManager.apply hands over (event_manager.py:219-240): an index tensor, `slice(None)` or None.
    `stones_cfg` names the stones' `RigidObjectCollection`: when the MDP regenerates stones (`binding(env,
    grid_bins=...)` or `intended_regen=True`), the stones of the reset envs are written to it (ENV:119-120), if the
    scene has it."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    b.ensure_pass1(env)
    if env_ids is None or isinstance(env_ids, slice):
        env_ids = torch.arange(env.num_envs, device=env.device)[env_ids if isinstance(env_ids, slice) else slice(None)]
    if len(env_ids) == 0:
        return
    b.mdp.reset(env.scene.env_origins, env_ids, b.buf, episode_length=env.episode_length_buf)
    k = len(env_ids)
    if write_to_sim and b.mdp.regenerates:
        from .env import write_stone_poses

        try:
            stones = env.scene[_entity_name(stones_cfg, "steps")]
        except KeyError:  # a scene without stone bodies: nothing to move
            stones = None
        if stones is not None:
            write_stone_poses(stones, b.mdp, env_ids)
    if write_to_sim:
        robot = env.scene[b.names[0]]
        root = b.buf.reset_root_state[:k]
        robot.write_root_pose_to_sim(root[:, :7], env_ids)
        robot.write_root_velocity_to_sim(root[:, 7:], env_ids)
        robot.write_joint_state_to_sim(b.buf.reset_joint_pos[:k], b.buf.reset_joint_vel[:k], None, env_ids)
    b.mdp.pass2(b.views(env), b.buf)
    b.open = False


# ---------------------------------------------------------------------------------------------- curriculum
def allsteps_level(env, env_ids, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> Dict[str, torch.Tensor]:
    """CurriculumManager term (logged under Curriculum/<name>/<key>, curriculum_manager.py:103-117): the current
    level and the statistic the promotion rule of ENV:471 looks at, as 0-dim device tensors (the manager's `reset()`
    does the `.item()` when it logs; computing the term itself does not synchronise).  The promotion itself happens
    inside `reset_allsteps`."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    s = b.mdp.stats_tensor  # int64 view of the device AsStats: 0 n_envs ... 8 sum_target_index ... 10 level
    n = torch.clamp(s[0], min=1).to(torch.float32)
    return {"level": s[10].to(torch.float32), "mean_target_index": s[8].to(torch.float32) / n}


def allsteps_grid(env, env_ids, asset_cfg=None, left_sensor_cfg=None, right_sensor_cfg=None) -> Dict[str, torch.Tensor]:
    """CurriculumManager term of the difficulty-grid curriculum (`binding(env, grid_bins=B)`): episodes ended so far
    (`attempts`), the share of them that passed half of their stones (`success_rate`) and the number of bins played at
    least once (`bins_visited`), as 0-dim device tensors read from the histograms in place -- no copy of the per-env
    bins, no synchronisation, no MDP pass.  The turnover itself happens inside `reset_allsteps`."""
    b = binding(env, asset_cfg, left_sensor_cfg, right_sensor_cfg)
    nb = b.mdp.grid_bins * b.mdp.grid_bins
    h = b.mdp.grid_hist_tensor
    att = h[:nb].to(torch.int64) & 0xFFFFFFFF  # (uint32 counters behind an int32 view)
    succ = h[256:256 + nb].to(torch.int64) & 0xFFFFFFFF
    total = att.sum()
    return {"attempts": total.to(torch.float32),
            "success_rate": succ.sum().to(torch.float32) / torch.clamp(total, min=1).to(torch.float32),
            "bins_visited": (att > 0).sum().to(torch.float32)}
