"""ctypes binding of include/allsteps_b200.h -- the stub a reference maintainer would add (INTEGRATION.md).

The shared library is built in-tree by `allsteps_isaaclab_b200.build` (nvcc, sm_100a only).  There is no
fallback: if the library is missing, `load()` raises, and every compute entry point returns an error on a
machine without a Blackwell device.
"""
from __future__ import annotations

import ctypes as C
import os

NUM_JOINTS = 21
NUM_STONES = 20  # AS_NUM_STONES: the default course length (AsParams.num_steps = 0)
MIN_STONES = 3   # AS_MIN_STONES
MAX_STONES = 32  # AS_MAX_STONES
OBS_DIM = 59
NUM_LEVELS = 10
ROOT_STATE_DIM = 13
NUM_REWARD_TERMS = 10
PEER_HANDLE_BYTES = 64  # AS_PEER_HANDLE_BYTES (sizeof(cudaIpcMemHandle_t))
TILE_ENVS = 128
ABI_VERSION = 5

FLAG_INTENDED_REGEN = 1 << 0
FLAG_SKIP_PASS2 = 1 << 1
FLAG_GRID_CURRICULUM = 1 << 2
FLAG_MISSED_STEP = 1 << 3
STEP_DEFER_FINISH = 1 << 0  # AsStepOut.flags

LIB_NAME = "liballsteps_b200.so"
LIB_PATH = os.environ.get("ALLSTEPS_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

_f = C.c_float
_i32 = C.c_int32
_i64 = C.c_int64
_ptr = C.c_void_p


class AsParams(C.Structure):
    _fields_ = [
        ("step_dt", _f), ("max_episode_length", _i32), ("step_radius", _f), ("dist_lower", _f),
        ("dist_upper", _f * NUM_LEVELS), ("yaw_range_deg", _f * 2), ("pitch_range_deg", _f * 2),
        ("init_step_separation", _f), ("max_level", _i32), ("termination_height", _f * NUM_LEVELS),
        ("applied_gain", _f * NUM_LEVELS), ("progress_threshold", _f), ("contact_epsilon", _f),
        ("stop_frames", _i32), ("energy_cost_scale", _f), ("actions_cost_scale", _f), ("alive_reward_scale", _f),
        ("dof_vel_scale", _f), ("joint_at_limit_cost_scale", _f), ("death_cost", _f),
        ("termination_height_absolute", _f), ("max_root_speed", _f), ("noise_span", _f), ("noise_lower", _f),
        ("clip_lower", _f), ("clip_upper", _f), ("default_root_pos", _f * 3),
        ("joint_lower", _f * NUM_JOINTS), ("joint_upper", _f * NUM_JOINTS), ("joint_gears", _f * NUM_JOINTS),
        ("reset_pose", _f * NUM_JOINTS), ("mirror_src", _i32 * NUM_JOINTS), ("mirror_sign", _f * NUM_JOINTS),
        ("missed_step_height", _f), ("flags", C.c_uint32), ("grid_bins", C.c_uint32), ("num_steps", C.c_uint32),
        ("seed", C.c_uint64),
    ]


class AsStateIn(C.Structure):
    _fields_ = [
        ("root_pos", _ptr), ("root_pos_stride", _i64),
        ("root_quat", _ptr), ("root_quat_stride", _i64),
        ("root_lin_vel", _ptr), ("root_lin_vel_stride", _i64),
        ("body_pos", _ptr), ("body_env_stride", _i64), ("body_row_stride", _i64),
        ("right_foot_row", _i32), ("left_foot_row", _i32), ("torso_row", _i32), ("quat_xyzw", _i32),
        ("joint_pos", _ptr), ("joint_pos_stride", _i64),
        ("joint_vel", _ptr), ("joint_vel_stride", _i64),
        ("contact_right", _ptr), ("contact_right_stride", _i64),
        ("contact_left", _ptr), ("contact_left_stride", _i64),
        ("env_origins", _ptr),
    ]


class AsStepOut(C.Structure):
    _fields_ = [("obs", _ptr), ("reward", _ptr), ("terminated", _ptr), ("time_out", _ptr), ("reward_terms", _ptr),
                ("dones", _ptr), ("obs_clip", _f), ("flags", C.c_uint32), ("final_obs", _ptr)]


class AsResetOut(C.Structure):
    _fields_ = [("root_state", _ptr), ("joint_pos", _ptr), ("joint_vel", _ptr), ("reset_ids", _ptr),
                ("n_reset", _ptr)]


class AsStats(C.Structure):
    _fields_ = [
        ("n_envs", _i64), ("n_reset", _i64), ("n_terminated", _i64), ("n_time_out", _i64), ("n_fell", _i64),
        ("n_so_fast", _i64), ("n_died", _i64), ("n_advanced", _i64), ("sum_target_index", _i64),
        ("n_regenerated", _i64), ("level", _i64), ("step_counter", _i64), ("sum_reward", C.c_double),
        ("n_missed", _i64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


STATS_ADDITIVE_FIELDS = 10  # leading int64 fields that are summed over ranks (AS_NUM_ADDITIVE_STATS)
MAX_GRID_CELLS = 256


class AsExchange(C.Structure):
    """What shards exchange per step: the statistics and this step's difficulty-grid outcomes (one device record)."""
    _fields_ = [("stats", AsStats), ("grid_attempts", C.c_uint32 * MAX_GRID_CELLS),
                ("grid_successes", C.c_uint32 * MAX_GRID_CELLS)]


STATS_INT64_WORDS = C.sizeof(AsStats) // 8          # int64 words of the AsStats head of an exchange record
EXCHANGE_INT64_WORDS = C.sizeof(AsExchange) // 8    # ... of the whole record (grid arrays: two uint32 per word)
# The handle's difficulty-grid histograms (uint32 attempts[256], then successes[256]) sit this many bytes behind the
# end of its exchange record in the workspace (a static_assert in csrc/as_internal.cuh holds the layout to it)
GRID_HIST_OFFSET = 1664


class AsMdpState(C.Structure):
    _fields_ = [("curr_target_index", _ptr), ("swing_leg", _ptr), ("target_reach_count", _ptr),
                ("episode_length", _ptr), ("curriculum", _ptr), ("potentials", _ptr), ("steps_pos", _ptr),
                ("steps_dphi", _ptr)]


class AsMirrorJob(C.Structure):
    _fields_ = [("in_", _ptr), ("out", _ptr), ("rows", _i64), ("kind", _i32), ("_pad", _i32)]


# name -> (restype, argtypes); every symbol the header declares
SIGNATURES = {
    "as_abi_version": (C.c_int, []),
    "as_last_error": (C.c_char_p, []),
    "as_workspace_bytes": (_i64, [_i64]),
    "as_workspace_bytes_for": (_i64, [C.POINTER(AsParams), _i64]),
    "as_create": (C.c_int, [C.POINTER(AsParams), _i64, _i64, C.c_int, _ptr, _i64, _ptr, C.POINTER(_ptr)]),
    "as_destroy": (None, [_ptr]),
    "as_generate_stones": (C.c_int, [_ptr, _ptr, _ptr, _i64, _ptr, _ptr]),
    "as_step_fused": (C.c_int, [_ptr, C.POINTER(AsStateIn), _ptr, _i64, C.POINTER(AsStepOut),
                                C.POINTER(AsResetOut), _ptr]),
    "as_step_pass1": (C.c_int, [_ptr, C.POINTER(AsStateIn), _ptr, _i64, _ptr, C.POINTER(AsStepOut), _ptr]),
    "as_reset": (C.c_int, [_ptr, _ptr, _ptr, _i64, _ptr, C.POINTER(AsResetOut), _ptr]),
    "as_step_pass2": (C.c_int, [_ptr, C.POINTER(AsStateIn), _ptr, _ptr]),
    "as_step_no_reset": (C.c_int, [_ptr, _ptr]),
    "as_stats_device_ptr": (C.c_int, [_ptr, C.POINTER(_ptr)]),
    "as_fold_stats": (C.c_int, [_ptr, _ptr]),
    "as_finish_step": (C.c_int, [_ptr, _ptr, _ptr]),
    "as_read_stats": (C.c_int, [_ptr, C.POINTER(AsStats), _ptr]),
    "as_apply_action": (C.c_int, [_ptr, _ptr, _i64, _ptr, _ptr]),
    "as_mirror_rows": (C.c_int, [_ptr, _ptr, _ptr, _i64, _i32, _ptr]),
    "as_mirror_batch": (C.c_int, [_ptr, C.POINTER(AsMirrorJob), _i32, _ptr]),
    "as_peer_create": (C.c_int, [_ptr, C.c_int, C.c_int, _ptr]),
    "as_peer_connect": (C.c_int, [_ptr, _ptr]),
    "as_peer_status": (C.c_int, [_ptr, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_i64), _ptr]),
    "as_global_stats_device_ptr": (C.c_int, [_ptr, C.POINTER(_ptr)]),
    "as_peer_three_call": (C.c_int, [_ptr, _i32]),
    "as_exchange_device_ptr": (C.c_int, [_ptr, C.POINTER(_ptr), C.POINTER(_ptr)]),
    "as_export_state": (C.c_int, [_ptr, C.POINTER(AsMdpState), _ptr]),
    "as_export_stone_poses": (C.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _ptr]),
    "as_import_state": (C.c_int, [_ptr, C.POINTER(AsMdpState), _ptr]),
    "as_snapshot_bytes": (_i64, [_ptr, _i32]),
    "as_snapshot": (C.c_int, [_ptr, _ptr, _i32, _ptr]),
    "as_restore": (C.c_int, [_ptr, _ptr, _i32, _ptr]),
    "as_grid_state": (C.c_int, [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "as_set_timing_events": (C.c_int, [_ptr, _ptr, _ptr]),
    "as_debug_timing": (C.c_int, [_ptr, _ptr, C.c_int, _ptr]),
    "as_launch_count": (_i64, [_ptr]),
    "as_sizeof": (_i64, [_i32]),
}

_lib = None


class AllstepsLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the in-tree CUDA library; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise AllstepsLibraryError(
            f"{LIB_PATH} is missing: build it with `python -m allsteps_isaaclab_b200.build` "
            "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for the Allsteps MDP step.")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.as_abi_version() != ABI_VERSION:
        raise AllstepsLibraryError(f"ABI mismatch: library {lib.as_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().as_last_error()
        raise AllstepsLibraryError(f"{what or 'allsteps call'} failed ({rc}): {msg.decode() if msg else ''}")
