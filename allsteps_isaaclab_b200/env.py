"""B1 face: the six `DirectRLEnv` hooks of the Allsteps task, delegating to the CUDA library.

`AllstepsHooksB200` is a mixin: put it in front of Isaac Lab's `DirectRLEnv` and it provides the hook methods of
the reference task (ENV = source/isaaclab_tasks/isaaclab_tasks/direct/allsteps/allsteps_env.py of the reference):

    class AllstepsEnv(AllstepsHooksB200, DirectRLEnv): ...

It reads exactly what the reference reads (`self.robot.data.*`, `self.sensor_left/right.data.force_matrix_w`,
`self.scene.env_origins`, `self.episode_length_buf`), performs the same three `robot.write_*_to_sim` calls, and keeps
the public attributes outside code touches (`right_body_indices`, `left_body_indices`, `negation_body_indices`,
`curr_target_index`, `curriculum`, `steps_pos`, ...).  The orchestration (`DirectRLEnv.step`, DRL:296-383) stays in
Isaac Lab.  `StandaloneAllstepsEnv` hosts the mixin without Isaac Lab (tests, synthetic physics): it replays the
post-physics part of `DirectRLEnv.step` (DRL:351-375) around the hooks.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .config import AllstepsCfg, JOINT_NAMES, NUM_JOINTS
from .mdp import AllstepsMDP, PhysicsViews, StepBuffers


def resolve_robot_tables(robot, cfg: AllstepsCfg):
    """What the reference resolves from the live articulation at run time (ENV:87-92, 287-291), checked against what
    the kernels assume: returns ((right_foot, left_foot, torso) body rows, joint limits (21,2) or None).

    The kernels' joint tables (gears CFG:133-155, reset pose ENV:505-511, mirror permutation CFG:217-219) are indexed in
    the PhysX joint order the reference documents; an articulation that enumerates its joints differently would be
    scaled, mirrored and actuated wrongly without any error, so a different order is refused here.  Joint limits are
    taken from `robot.data.joint_pos_limits` (what ENV:287-291 reads; PhysX' own degree -> radian conversion need not
    round like the table's) and must not differ between envs (they are O(1) constants of the kernels)."""
    names = list(robot.data.body_names)
    body_rows = (names.index(cfg.foot_names[0]), names.index(cfg.foot_names[1]), names.index(cfg.torso_name))
    jn = list(robot.data.joint_names)
    if jn != list(JOINT_NAMES):
        raise ValueError("robot.data.joint_names differs from the joint order the Allsteps kernels are built for "
                         f"(CFG:133-155):\n  robot:   {jn}\n  kernels: {list(JOINT_NAMES)}")
    limits = getattr(robot.data, "joint_pos_limits", None)
    if limits is None:
        return body_rows, None
    limits = torch.as_tensor(limits)
    if limits.dim() != 3 or tuple(limits.shape[1:]) != (NUM_JOINTS, 2):
        raise ValueError(f"robot.data.joint_pos_limits must be (N,{NUM_JOINTS},2), got {tuple(limits.shape)}")
    if limits.shape[0] > 1 and not bool((limits == limits[:1]).all()):
        raise ValueError("robot.data.joint_pos_limits differ between envs; the Allsteps kernels take one limit table")
    return body_rows, limits[0].detach().to(torch.float32).cpu()


def write_stone_poses(steps, mdp: AllstepsMDP, env_ids: torch.Tensor):
    """ENV:119-120: the stones of `env_ids` as the MDP holds them, written to the simulator's stone collection
    (`RigidObjectCollection.write_object_pose_to_sim`, poses (k,S,7): position + identity quaternion w,x,y,z; S is the
    course length `mdp.num_steps`)."""
    pos = mdp.export_state(("steps_pos",))["steps_pos"][env_ids]
    quat = torch.tensor([1.0, 0.0, 0.0, 0.0], device=pos.device).expand(pos.shape[0], mdp.num_steps, 4)
    steps.write_object_pose_to_sim(torch.cat((pos, quat), dim=-1), env_ids)  # ENV:119-120


class AllstepsHooksB200:
    """Hook methods of `AllstepsEnv(DirectRLEnv)` (ENV:34) backed by `AllstepsMDP`."""

    def _init_allsteps_b200(self, task_cfg: Optional[AllstepsCfg] = None, seed: int = 0, final_obs: bool = False,
                            distributed: bool = False, **mdp_kwargs):
        """Call at the end of `__init__` (replaces ENV:40-102).

        final_obs: publish `extras["final_obs"]` (N,59) every step: for the envs that reset in the step (`reset_buf`),
        the observation of the state their episode ended in -- `obs` holds their start pose -- so that a time-out can
        be bootstrapped with `gamma * V(final_obs)`.  Rows of the other envs hold whatever an earlier step left there.

        distributed: one process per GPU under torch.distributed (torchrun), this env holding one shard of the run's
        envs.  The shard's global env ids follow the other ranks' (so draws do not depend on the number of GPUs) and
        the handle runs in the global 3-call mode: promotion, "did any env reset" and the grid histograms over all
        shards, bit-identical to one env holding all of them (`AllstepsMDP.connect_peers(three_call=True)`)."""
        self.task_cfg = task_cfg or AllstepsCfg()
        dev = torch.device(self.device)
        body_rows, joint_limits = resolve_robot_tables(self.robot, self.task_cfg)
        if distributed:
            from .sharding import global_env_offset

            mdp_kwargs["env_id_offset"] = global_env_offset(self.num_envs, dev)
        self.mdp = AllstepsMDP(self.num_envs, device=dev, cfg=self.task_cfg, seed=seed, joint_limits=joint_limits,
                               **mdp_kwargs)
        if distributed:
            self.mdp.connect_peers(three_call=True)
        self.buf = StepBuffers(self.num_envs, dev, reward_terms=True, final_obs=final_obs)
        self.foot_indices = [body_rows[0], body_rows[1]]  # ENV:87
        self.torso_index = body_rows[2]  # ENV:88
        jn = list(self.robot.data.joint_names)
        as_idx = lambda ns: torch.tensor([jn.index(n) for n in ns], dtype=torch.int64, device=dev)  # noqa: E731
        self.right_body_indices = as_idx(self.task_cfg.right_body_names)  # ENV:90
        self.left_body_indices = as_idx(self.task_cfg.left_body_names)  # ENV:91
        self.negation_body_indices = as_idx(self.task_cfg.negation_body_names)  # ENV:92
        self.num_steps = self.mdp.num_steps  # CFG:90, the course length the kernels run
        self.actions = torch.zeros(self.num_envs, 21, device=dev)
        self._pass_epoch = -1
        self._generate_foot_steps()  # ENV:71

    # ------------------------------------------------------------------ views of the PhysX-side tensors
    def _physics_views(self) -> PhysicsViews:
        d = self.robot.data
        t = (d.root_pos_w, d.root_quat_w, d.root_lin_vel_w, d.body_pos_w, d.joint_pos, d.joint_vel,
             self.sensor_right.data.force_matrix_w, self.sensor_left.data.force_matrix_w, self.scene.env_origins)
        return PhysicsViews.cached(self, t, (self.foot_indices[0], self.foot_indices[1], self.torso_index))

    # ------------------------------------------------------------------ ENV:106-123
    def _generate_foot_steps(self, env_ids: Optional[torch.Tensor] = None):
        self.mdp.generate_stones(self.scene.env_origins, env_ids)
        self._write_stone_poses(env_ids if env_ids is not None else torch.arange(self.num_envs, device=self.device))

    def _write_stone_poses(self, env_ids: torch.Tensor):
        """The stones of `env_ids` to the `steps` collection, when the env has one (built by `_setup_scene`)."""
        steps = getattr(self, "steps", None)
        if steps is not None and hasattr(steps, "write_object_pose_to_sim"):
            write_stone_poses(steps, self.mdp, env_ids)

    # ------------------------------------------------------------------ the six hooks
    def _pre_physics_step(self, actions: torch.Tensor):  # ENV:257-268 (the clamp is applied inside the kernels)
        self.actions = actions.to(torch.float32)
        self._efforts_valid = False

    def _apply_action(self):  # ENV:270-274
        # DirectRLEnv.step calls this `decimation` = 4 times per env step (DRL:333-349) with the same actions and the
        # same curriculum levels -- both change only outside that loop (`_pre_physics_step`, `_reset_idx`): the
        # efforts are computed by the first call and handed out again by the other three
        if not getattr(self, "_efforts_valid", False):
            self._efforts = self.mdp.apply_action(self.actions, getattr(self, "_efforts", None))
            self._efforts_valid = True
        self.robot.set_joint_effort_target(self._efforts)

    def _get_dones(self):  # ENV:396-405; the same launch produces the rewards of ENV:347-394
        self._efforts_valid = False  # (levels can change from here on)
        self.mdp.pass1(self._physics_views(), self.actions, self.buf, episode_length=self.episode_length_buf)
        self._pass1_open = True  # closed by `_reset_idx` (pass 2) or, when nothing resets, by `_get_observations`
        return self.buf.terminated, self.buf.time_out

    def _get_rewards(self) -> torch.Tensor:  # ENV:347-394 (computed against the `terminated` returned above)
        return self.buf.reward

    def _reset_idx(self, env_ids: Optional[torch.Tensor]):  # ENV:469-567
        if env_ids is None or len(env_ids) == self.num_envs:
            env_ids = self.robot._ALL_INDICES
        self._efforts_valid = False
        self.robot.reset(env_ids)
        super()._reset_idx(env_ids)  # scene.reset (contact rows -> 0) and episode_length_buf[env_ids] = 0, DRL:563-584
        self.mdp.reset(self.scene.env_origins, env_ids, self.buf)
        if self.mdp.regenerates:
            # ENV:497-500 -> ENV:119-120: stones regenerated by the reset go to PhysX.  All rows of the reset envs are
            # written, also those intended regeneration left as they were (same values; cheaper than a host sync
            # to learn which ones changed)
            self._write_stone_poses(env_ids)
        k = len(env_ids)
        root = self.buf.reset_root_state[:k]
        self.robot.write_root_pose_to_sim(root[:, :7], env_ids)  # ENV:563
        self.robot.write_root_velocity_to_sim(root[:, 7:], env_ids)  # ENV:564
        self.robot.write_joint_state_to_sim(self.buf.reset_joint_pos[:k], self.buf.reset_joint_vel[:k], None,
                                            env_ids)  # ENV:565
        self.mdp.pass2(self._physics_views(), self.buf)  # ENV:567
        self._pass1_open = False

    def _get_observations(self) -> Dict[str, torch.Tensor]:  # ENV:326-345
        if getattr(self, "_pass1_open", False):  # DRL:360 skipped `_reset_idx`: no pass 2 this step
            self.mdp.no_reset()
            self._pass1_open = False
        if self.buf.final_obs is not None:
            self.extras["final_obs"] = self.buf.final_obs
        return {"policy": self.buf.obs}

    # ------------------------------------------------------------------ the reference's public buffers, on demand
    def _state(self, field: str) -> torch.Tensor:
        return self.mdp.export_state((field,))[field]  # (only the buffer that was asked for is materialised)

    curr_target_index = property(lambda self: self._state("curr_target_index"))
    prev_target_index = property(lambda self: self._state("prev_target_index"))
    next_target_index = property(lambda self: self._state("next_target_index"))
    swing_leg = property(lambda self: self._state("swing_leg"))
    target_reach_count = property(lambda self: self._state("target_reach_count"))
    curriculum = property(lambda self: self._state("curriculum"))
    potentials = property(lambda self: self._state("potentials"))
    steps_pos = property(lambda self: self._state("steps_pos"))
    steps_dphi = property(lambda self: self._state("steps_dphi"))


class _StandaloneBase:
    """What the mixin needs from `DirectRLEnv` when Isaac Lab is absent: `_reset_idx` side effects, DRL:563-584."""

    def _reset_idx(self, env_ids):
        self.sensor_left.data.force_matrix_w[env_ids] = 0.0  # contact_sensor.py:155 via scene.reset
        self.sensor_right.data.force_matrix_w[env_ids] = 0.0
        self.episode_length_buf[env_ids] = 0  # DRL:584


class StandaloneAllstepsEnv(AllstepsHooksB200, _StandaloneBase):
    """The hooks hosted on plain tensor holders (`robot`, `sensor_left/right`, `scene`): a `DirectRLEnv` stand-in that
    runs the post-physics section of `DirectRLEnv.step` (DRL:351-375).  Physics is whatever the caller installs."""

    def __init__(self, robot, sensor_left, sensor_right, scene, device, task_cfg: Optional[AllstepsCfg] = None,
                 seed: int = 0, **mdp_kwargs):
        self.robot, self.sensor_left, self.sensor_right, self.scene = robot, sensor_left, sensor_right, scene
        self.device = device
        self.num_envs = scene.env_origins.shape[0]
        dev = torch.device(device)
        self.episode_length_buf = torch.zeros(self.num_envs, dtype=torch.long, device=dev)  # DRL:179
        self.reset_terminated = torch.zeros(self.num_envs, dtype=torch.bool, device=dev)  # DRL:180
        self.reset_time_outs = torch.zeros(self.num_envs, dtype=torch.bool, device=dev)  # DRL:181
        self.reset_buf = torch.zeros(self.num_envs, dtype=torch.bool, device=dev)  # DRL:182
        self.common_step_counter = 0
        self.extras = {}
        self._init_allsteps_b200(task_cfg, seed, **mdp_kwargs)

    def reset(self):
        """DRL:256-279: `_reset_idx(all ids)` before any step, then the observations (no physics here)."""
        self._reset_idx(torch.arange(self.num_envs, dtype=torch.int64, device=self.episode_length_buf.device))
        self.obs_buf = self._get_observations()
        return self.obs_buf, self.extras

    def post_physics_step(self, actions: torch.Tensor):
        """DRL:326 + DRL:351-375."""
        self._pre_physics_step(actions)
        self.episode_length_buf += 1
        self.common_step_counter += 1
        terminated, time_outs = self._get_dones()
        self.reset_terminated[:], self.reset_time_outs[:] = terminated, time_outs
        self.reset_buf = self.reset_terminated | self.reset_time_outs
        self.reward_buf = self._get_rewards()
        reset_env_ids = self.reset_buf.nonzero(as_tuple=False).squeeze(-1)
        if len(reset_env_ids) > 0:
            self._reset_idx(reset_env_ids)
        self.obs_buf = self._get_observations()
        return self.obs_buf, self.reward_buf, self.reset_terminated, self.reset_time_outs, self.extras
