"""Term configurations for Isaac Lab's managers (B2 face, SURVEY 8b): the Allsteps MDP as a manager-based task.

`build_manager_cfgs()` returns the five configuration dictionaries the reference's managers take --

    ObservationManager(cfgs["observations"], env)   group "policy": 7 terms, concatenated = the 59 columns of ENV:326-345
    RewardManager(cfgs["rewards"], env)             one term with weight 1 / step_dt (reward_manager.py:148 multiplies
                                                    by weight * dt), or the ten terms of ENV:350-375 (`per_term=True`)
    TerminationManager(cfgs["terminations"], env)   fell | so_fast | died, and the time-out with `time_out=True`
    EventManager(cfgs["events"], env)               `reset_allsteps` in mode "reset" (ENV:469-567)
    CurriculumManager(cfgs["curriculum"], env)      `allsteps_level` (logging; the promotion happens in the reset),
                                                    and `allsteps_grid` with `grid_curriculum=True`

-- built from the cfg classes of the `isaaclab.managers` module that is passed in (default: the installed Isaac Lab).
Every term's scene entities are named by `SceneEntityCfg` params, which `ManagerBase._resolve_common_term_cfg`
(manager_base.py:219-298) resolves against `env.scene` and checks against the term's signature.
"""
from __future__ import annotations

import importlib
from typing import Any, Dict

from . import terms
from .config import AllstepsCfg


def build_manager_cfgs(managers=None, robot: str = "robot", left_sensor: str = "foot_contacts_left",
                       right_sensor: str = "foot_contacts_right", task_cfg: AllstepsCfg | None = None,
                       per_term_rewards: bool = False, grid_curriculum: bool = False) -> Dict[str, Any]:
    """grid_curriculum: also log the difficulty-grid curriculum through the `allsteps_grid` curriculum term.  The grid
    itself is switched on where the MDP is made: `terms.binding(env, grid_bins=B)` before the managers are built."""
    M = managers if managers is not None else importlib.import_module("isaaclab.managers")
    cfg = task_cfg or AllstepsCfg()

    def ent():  # fresh objects per term: the managers write the resolved indices into them
        return {"asset_cfg": M.SceneEntityCfg(robot), "left_sensor_cfg": M.SceneEntityCfg(left_sensor),
                "right_sensor_cfg": M.SceneEntityCfg(right_sensor)}

    policy = M.ObservationGroupCfg()
    policy.concatenate_terms = True
    policy.enable_corruption = False
    for fn in terms.OBSERVATION_TERMS:  # cfg order = column order of ENV:330-343
        setattr(policy, fn.__name__, M.ObservationTermCfg(func=fn, params=ent()))
    observations = {"policy": policy}

    inv_dt = 1.0 / cfg.step_dt
    if per_term_rewards:
        signs = {"alive": 1.0, "progress": 1.0, "step_reward": 1.0, "target_bonus": 1.0}
        rewards = {name: M.RewardTermCfg(func=terms.reward_term, weight=signs.get(name, -1.0) * inv_dt,
                                         params={"name": name, **ent()}) for name in terms.REWARD_COLUMNS}
    else:
        rewards = {"allsteps": M.RewardTermCfg(func=terms.allsteps_total_reward, weight=inv_dt, params=ent())}

    terminations = {
        "terminated": M.TerminationTermCfg(func=terms.allsteps_terminated, params=ent()),
        "time_out": M.TerminationTermCfg(func=terms.allsteps_time_out, params=ent(), time_out=True),
    }
    events = {"reset_allsteps": M.EventTermCfg(func=terms.reset_allsteps, mode="reset", params=ent())}
    curriculum = {"allsteps_level": M.CurriculumTermCfg(func=terms.allsteps_level, params=ent())}
    if grid_curriculum:
        curriculum["allsteps_grid"] = M.CurriculumTermCfg(func=terms.allsteps_grid, params=ent())
    return {"observations": observations, "rewards": rewards, "terminations": terminations, "events": events,
            "curriculum": curriculum}
