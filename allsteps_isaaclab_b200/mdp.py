"""`AllstepsMDP` -- host-side owner of the Allsteps-v0 MDP state on one GPU.

It holds what `AllstepsEnv.__init__` allocates in the reference (ENV:41-96) -- but as one packed device
workspace -- and exposes the step of direct_rl_env.py:351-375 as `step()` (one fused launch) or as
`pass1() / reset() / pass2()` for hosts that run PhysX in between.  PyTorch is used for device memory and
streams only; every number is produced by the CUDA library behind include/allsteps_b200.h.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch

from . import _cabi
from .config import AllstepsCfg, NUM_JOINTS, OBS_DIM
from .params import make_params


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require(t: torch.Tensor, dtype, device, name: str):
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if t.device != device:
        raise ValueError(f"{name}: expected device {device}, got {t.device}")


class PhysicsViews:
    """Device views of the PhysX-side tensors of one step, in the layouts Isaac Lab publishes them.

    Accepts the tensors the reference reads (`robot.data.root_pos_w`, ..., `sensor_left.data.force_matrix_w`);
    strided views such as slices of `root_state_w (N,13)` / `body_state_w (N,B,13)` are taken as they are.

    The contact matrices are (N,1,S,3), S the course length (`AllstepsCfg.num_steps`, 3..32); `num_steps` records it,
    and the MDP refuses views whose S is not its own.

    The two contact matrices may also be PINNED HOST tensors: under unified addressing they are device-accessible,
    and since the step needs only the current stone's 12-byte vector per foot and env (24 of 480 bytes), letting the
    gather kernel fetch those through PCIe beats copying the matrices (bench.py e2e: 11.4 vs 16.1 ms per step at 1 M
    envs).
    """

    def __init__(self, *, root_pos_w, root_quat_w, root_lin_vel_w, body_pos_w, joint_pos, joint_vel,
                 force_matrix_right, force_matrix_left, env_origins, body_rows=(0, 1, 2), quat_xyzw=False):
        self.tensors = dict(root_pos_w=root_pos_w, root_quat_w=root_quat_w, root_lin_vel_w=root_lin_vel_w,
                            body_pos_w=body_pos_w, joint_pos=joint_pos, joint_vel=joint_vel,
                            force_matrix_right=force_matrix_right, force_matrix_left=force_matrix_left,
                            env_origins=env_origins)
        N = root_pos_w.shape[0]
        s = _cabi.AsStateIn()

        def rows(t, width, name):
            if t.dtype != torch.float32:
                raise TypeError(f"{name} must be float32")
            if t.dim() != 2 or t.shape[0] != N or t.shape[1] != width or (N > 1 and t.stride(1) != 1):
                raise ValueError(f"{name} must be a (N,{width}) view with unit inner stride, got {tuple(t.shape)}")
            return t.data_ptr(), (t.stride(0) if N > 1 else width)

        s.root_pos, s.root_pos_stride = rows(root_pos_w, 3, "root_pos_w")
        s.root_quat, s.root_quat_stride = rows(root_quat_w, 4, "root_quat_w")
        s.root_lin_vel, s.root_lin_vel_stride = rows(root_lin_vel_w, 3, "root_lin_vel_w")
        s.joint_pos, s.joint_pos_stride = rows(joint_pos, NUM_JOINTS, "joint_pos")
        s.joint_vel, s.joint_vel_stride = rows(joint_vel, NUM_JOINTS, "joint_vel")
        if body_pos_w.dim() != 3 or body_pos_w.shape[0] != N or body_pos_w.shape[2] != 3 or body_pos_w.stride(2) != 1:
            raise ValueError("body_pos_w must be a (N,B,3) view with unit inner stride")
        B = body_pos_w.shape[1]
        s.body_pos = body_pos_w.data_ptr()
        s.body_env_stride = body_pos_w.stride(0) if N > 1 else B * 3
        s.body_row_stride = body_pos_w.stride(1) if B > 1 else 3
        s.right_foot_row, s.left_foot_row, s.torso_row = (int(b) for b in body_rows)
        s.quat_xyzw = 1 if quat_xyzw else 0  # PhysX' own order; Isaac Lab's root_quat_w is w,x,y,z
        if max(body_rows) >= B:
            raise ValueError("body row index out of range")
        S = force_matrix_right.shape[-2] if force_matrix_right.dim() >= 3 else -1
        for name, t in (("force_matrix_right", force_matrix_right), ("force_matrix_left", force_matrix_left)):
            if (t.dtype != torch.float32 or t.dim() < 3 or t.shape[0] != N or t.shape[-1] != 3 or t.shape[-2] != S
                    or not _cabi.MIN_STONES <= S <= _cabi.MAX_STONES):
                raise ValueError(f"{name} must be float32 (N,1,S,3) with S in {_cabi.MIN_STONES}..{_cabi.MAX_STONES}, "
                                 f"the same S for both feet; got {tuple(t.shape)}")
            if not t[0].is_contiguous():
                raise ValueError(f"{name}: the per-env (1,S,3) block must be contiguous")
            if t.device.type == "cpu" and root_pos_w.device.type == "cuda" and not t.is_pinned():
                raise ValueError(f"{name}: a host tensor must be pinned (page-locked) to be read by the device")
        s.contact_right = force_matrix_right.data_ptr()
        s.contact_right_stride = force_matrix_right.stride(0) if N > 1 else S * 3
        s.contact_left = force_matrix_left.data_ptr()
        s.contact_left_stride = force_matrix_left.stride(0) if N > 1 else S * 3
        if env_origins is not None:
            if env_origins.dtype != torch.float32 or tuple(env_origins.shape) != (N, 3) or not env_origins.is_contiguous():
                raise ValueError("env_origins must be contiguous float32 (N,3)")
            s.env_origins = env_origins.data_ptr()
        self.struct = s
        self.num_envs = N
        self.num_steps = S
        self.device = root_pos_w.device

    _FIELDS = ("root_pos_w", "root_quat_w", "root_lin_vel_w", "body_pos_w", "joint_pos", "joint_vel",
               "force_matrix_right", "force_matrix_left", "env_origins")

    @classmethod
    def cached(cls, holder, tensors: tuple, body_rows, quat_xyzw: bool = False) -> "PhysicsViews":
        """The views of `tensors` (in `_FIELDS` order), rebuilt -- struct and validation -- only when an address,
        stride, shape or dtype changed since the last call with this `holder`.  Isaac Lab's data properties hand out
        fresh views of persistent PhysX-side buffers on every access; the hooks ask for them two or three times a step."""
        key = tuple((t.data_ptr(), t.stride(), t.shape, t.dtype) for t in tensors) + (tuple(body_rows), quat_xyzw)
        v = getattr(holder, "_as_views", None)
        if v is None or holder._as_views_key != key:
            v = cls(**dict(zip(cls._FIELDS, tensors)), body_rows=body_rows, quat_xyzw=quat_xyzw)
            holder._as_views, holder._as_views_key = v, key
        else:
            v.tensors = dict(zip(cls._FIELDS, tensors))  # (keep THESE tensor objects alive while kernels run)
        return v

    @classmethod
    def from_dict(cls, d: Dict[str, torch.Tensor], env_origins, body_rows=(0, 1, 2), quat_xyzw=False) -> "PhysicsViews":
        return cls(root_pos_w=d["root_pos_w"], root_quat_w=d["root_quat_w"], root_lin_vel_w=d["root_lin_vel_w"],
                   body_pos_w=d["body_pos_w"], joint_pos=d["joint_pos"], joint_vel=d["joint_vel"],
                   force_matrix_right=d["force_matrix_right"], force_matrix_left=d["force_matrix_left"],
                   env_origins=env_origins, body_rows=body_rows, quat_xyzw=quat_xyzw)


class StepBuffers:
    """Output tensors of a step; allocated once, overwritten every step (the caller clones what it keeps)."""

    def __init__(self, num_envs: int, device, reward_terms: bool = False, reset_rows: bool = True,
                 obs_clip: float = 0.0, final_obs: bool = False):
        """obs_clip > 0: `obs` comes out clamped to +-obs_clip, the `clip_obs` of RlGamesVecEnvWrapper._process_obs
        (isaaclab_rl/rl_games.py:293) folded into the kernel's observation write; 0 keeps the raw ENV:326-345 values.
        final_obs: also allocate `final_obs` (N,59), where every step writes the observation of the state an env's
        episode ended in, at the rows of the envs that reset (`dones`) and clamped like `obs` -- what bootstrapping a
        time-out needs, since `obs` holds the start pose of those envs.  Other rows keep what they held."""
        kw = dict(device=device)
        self.obs_clip = float(obs_clip)
        self.obs = torch.empty(num_envs, OBS_DIM, dtype=torch.float32, **kw)
        self.reward = torch.empty(num_envs, dtype=torch.float32, **kw)
        self.terminated = torch.zeros(num_envs, dtype=torch.bool, **kw)
        self.time_out = torch.zeros(num_envs, dtype=torch.bool, **kw)
        self.dones = torch.zeros(num_envs, dtype=torch.bool, **kw)  # terminated | time_out (reset_buf)
        self.reward_terms = (torch.empty(num_envs, _cabi.NUM_REWARD_TERMS, dtype=torch.float32, **kw)
                             if reward_terms else None)
        self.reset_root_state = self.reset_joint_pos = self.reset_joint_vel = None
        self.reset_ids = self.n_reset = None
        if reset_rows:
            self.reset_root_state = torch.zeros(num_envs, _cabi.ROOT_STATE_DIM, dtype=torch.float32, **kw)
            self.reset_joint_pos = torch.zeros(num_envs, NUM_JOINTS, dtype=torch.float32, **kw)
            self.reset_joint_vel = torch.zeros(num_envs, NUM_JOINTS, dtype=torch.float32, **kw)
            self.reset_ids = torch.zeros(num_envs, dtype=torch.int32, **kw)
            self.n_reset = torch.zeros(1, dtype=torch.int32, **kw)
        self.final_obs = torch.zeros(num_envs, OBS_DIM, dtype=torch.float32, **kw) if final_obs else None
        self.step_out = _cabi.AsStepOut(_ptr(self.obs), _ptr(self.reward), _ptr(self.terminated),
                                        _ptr(self.time_out), _ptr(self.reward_terms), _ptr(self.dones),
                                        self.obs_clip, 0, _ptr(self.final_obs))
        self.reset_out = _cabi.AsResetOut(_ptr(self.reset_root_state), _ptr(self.reset_joint_pos),
                                          _ptr(self.reset_joint_vel), _ptr(self.reset_ids), _ptr(self.n_reset))


class CapturedStep:
    """A fused step captured as a CUDA graph (see AllstepsMDP.capture_step)."""

    def __init__(self, mdp: "AllstepsMDP", views: PhysicsViews, actions: torch.Tensor, out: StepBuffers,
                 global_stats: Optional[torch.Tensor] = None):
        self.mdp = mdp
        self.keep = (views, actions, out, global_stats)
        self.graph = torch.cuda.CUDAGraph()
        before = mdp.launch_count
        with torch.cuda.device(mdp.device):
            with torch.cuda.graph(self.graph):  # stream capture: the kernels are recorded, not executed
                mdp.step(views, actions, out, global_stats)
        self.kernels_per_replay = mdp.launch_count - before

    def replay(self):
        self.graph.replay()


class AllstepsMDP:
    def __init__(self, num_envs: int, device="cuda:0", cfg: Optional[AllstepsCfg] = None, seed: int = 0,
                 env_id_offset: int = 0, intended_regen: bool = False, skip_pass2: bool = False,
                 grid_bins: int = 0, joint_limits: Optional[torch.Tensor] = None, missed_step: bool = False):
        """joint_limits: optional (21,2) [lower, upper] in radians as the simulator reports them
        (`robot.data.joint_pos_limits[0]`, ENV:287-291); default = the MJCF table of config.py."""
        self.lib = _cabi.load()  # raises if the CUDA library was not built: there is no fallback
        self.cfg = cfg or AllstepsCfg()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _cabi.AllstepsLibraryError("AllstepsMDP runs on a CUDA device only (sm_100a); no CPU path exists")
        self.num_envs = int(num_envs)
        self.env_id_offset = int(env_id_offset)
        flags = (_cabi.FLAG_INTENDED_REGEN if intended_regen else 0) | (_cabi.FLAG_SKIP_PASS2 if skip_pass2 else 0)
        flags |= _cabi.FLAG_GRID_CURRICULUM if grid_bins else 0
        flags |= _cabi.FLAG_MISSED_STEP if missed_step else 0  # extension: AllstepsCfg.missed_step_height
        self.grid_bins = int(grid_bins)
        self.seed = int(seed)
        self.params = make_params(self.cfg, seed=seed, flags=flags, grid_bins=self.grid_bins,
                                  joint_limits=joint_limits)
        self.num_steps = int(self.params.num_steps) or _cabi.NUM_STONES  # S, stones per course (CFG:90; 0: default)
        nbytes = self.lib.as_workspace_bytes_for(C.byref(self.params), self.num_envs)
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            assert self.workspace.data_ptr() % 256 == 0
            handle = C.c_void_p()
            _cabi.check(self.lib.as_create(C.byref(self.params), self.num_envs, self.env_id_offset,
                                           self.device.index or 0, self.workspace.data_ptr(), nbytes,
                                           self._stream(), C.byref(handle)), "as_create")
        self.handle = handle
        stats_ptr = C.c_void_p()
        _cabi.check(self.lib.as_stats_device_ptr(self.handle, C.byref(stats_ptr)), "as_stats_device_ptr")
        off = stats_ptr.value - self.workspace.data_ptr()
        # device view of the folded step statistics (int64 fields; see _cabi.AsStats)
        self.stats_tensor = self.workspace[off: off + C.sizeof(_cabi.AsStats)].view(torch.int64)
        # ... and of the whole exchange record it heads (statistics + this step's difficulty-grid outcomes): what a
        # sharded caller all-reduces -- `exchange_tensor[:10]` and, with the grid curriculum, `exchange_tensor[grid_words]`
        # (two uint32 counters per int64 word; the sums cannot carry) -- and hands to `finish_step`
        self.exchange_tensor = self.workspace[off: off + C.sizeof(_cabi.AsExchange)].view(torch.int64)
        self.grid_words = slice(_cabi.STATS_INT64_WORDS, _cabi.EXCHANGE_INT64_WORDS)
        # ... and of the difficulty-grid histograms: attempts in [:256], successes in [256:] (bin b = pitch bin *
        # grid_bins + yaw bin; uint32 counters read as int32) -- what a logger reads without a copy or a synchronisation
        h0 = off + C.sizeof(_cabi.AsExchange) + _cabi.GRID_HIST_OFFSET
        self.grid_hist_tensor = self.workspace[h0: h0 + 8 * _cabi.MAX_GRID_CELLS].view(torch.int32)
        # every env that resets may get new stones (grid curriculum, intended regeneration): a host that keeps the
        # stones in a simulator must write them there after each reset
        self.regenerates = bool(flags & (_cabi.FLAG_GRID_CURRICULUM | _cabi.FLAG_INTENDED_REGEN))
        self._keepalive = None

    # ------------------------------------------------------------------ plumbing
    def _stream(self) -> int:
        # (the raw handle of torch's current stream on this device: the private accessor is an order of magnitude
        # cheaper than building a torch.cuda.Stream object on every library call)
        raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
        if raw is not None:
            return raw(self.device.index if self.device.index is not None else torch.cuda.current_device())
        return torch.cuda.current_stream(self.device).cuda_stream

    def __del__(self):
        h = getattr(self, "handle", None)
        if h is not None and h.value:
            self.lib.as_destroy(h)
            self.handle = None

    @property
    def launch_count(self) -> int:
        return int(self.lib.as_launch_count(self.handle))

    def _check_views(self, views: PhysicsViews):
        if views.num_envs != self.num_envs:
            raise ValueError("views belong to a different number of envs")
        if views.num_steps != self.num_steps:
            raise ValueError(f"contact matrices are (N,1,{views.num_steps},3); this MDP runs courses of "
                             f"num_steps={self.num_steps} stones")

    # ------------------------------------------------------------------ stones (ENV:106-174)
    def generate_stones(self, env_origins: torch.Tensor, env_ids: Optional[torch.Tensor] = None,
                        uniforms: Optional[torch.Tensor] = None):
        _require(env_origins, torch.float32, self.device, "env_origins")
        ids_ptr, n_ids = None, 0
        if env_ids is not None:
            env_ids = env_ids.to(device=self.device, dtype=torch.int32).contiguous()
            ids_ptr, n_ids = env_ids.data_ptr(), env_ids.numel()
        if uniforms is not None:
            _require(uniforms, torch.float32, self.device, "uniforms")
            if tuple(uniforms.shape) not in ((5, self.num_envs, self.num_steps), (3, self.num_envs, self.num_steps)):
                raise ValueError(f"uniforms must be (5|3, N, S) with S = num_steps = {self.num_steps}")
            uniforms = uniforms.contiguous()
        _cabi.check(self.lib.as_generate_stones(self.handle, env_origins.data_ptr(), ids_ptr, n_ids,
                                                _ptr(uniforms), self._stream()), "as_generate_stones")

    # ------------------------------------------------------------------ fused step (DRL:351-375)
    def step(self, views: PhysicsViews, actions: torch.Tensor, out: StepBuffers,
             global_stats: Optional[torch.Tensor] = None, finish: bool = True):
        """One MDP step in one fused launch. Results land in `out`; nothing is synchronised."""
        self._check_views(views)
        _require(actions, torch.float32, self.device, "actions")
        if actions.dim() != 2 or actions.shape != (self.num_envs, NUM_JOINTS) or actions.stride(1) != 1:
            raise ValueError("actions must be (N,21) with unit inner stride")
        stride = actions.stride(0) if self.num_envs > 1 else NUM_JOINTS
        # finish=False announces as_fold_stats + an all-reduce + as_finish_step(global): the step must stay open
        out.step_out.flags = 0 if finish else _cabi.STEP_DEFER_FINISH
        _cabi.check(self.lib.as_step_fused(self.handle, C.byref(views.struct), actions.data_ptr(), stride,
                                           C.byref(out.step_out), C.byref(out.reset_out), self._stream()),
                    "as_step_fused")
        self._keepalive = (views, actions, out)
        if finish:
            self.finish_step(global_stats)

    def capture_step(self, views: PhysicsViews, actions: torch.Tensor, out: StepBuffers,
                     global_stats: Optional[torch.Tensor] = None) -> "CapturedStep":
        """Record one fused step (all its launches) into a CUDA graph bound to these buffers.  Replaying costs one
        graph launch instead of several library calls -- what matters at 4 K..64 K envs, where the step is
        launch-latency bound.  The producer of the physics tensors must write into the same storage every step."""
        return CapturedStep(self, views, actions, out, global_stats)

    # ------------------------------------------------------------------ cross-shard promotion over NVLink peer memory
    def connect_peers(self, group=None, three_call: bool = False):
        """One process per GPU, every rank owning one env-id shard: after this call `step()` / `finish_step()` decide
        the promotion rule (ENV:471) and the "did any env reset" test (DRL:359) on the sum over ALL shards.  The sum is
        formed by one small kernel that stores this shard's ten step counters into every peer's exchange buffer
        through NVLink and reads theirs -- no NCCL call on the step path.  torch.distributed is used once, here, to
        hand round the 64-byte CUDA IPC handles.  Every rank must step in lockstep from now on.

        three_call: the same for the 3-call path (`pass1` / `reset` / `pass2` / `no_reset`, what the Isaac Lab faces
        drive) instead of `step()`: promotion, "did any env reset" and the grid histograms over all shards, one exchange
        per `pass1`.  Every rank must make the same sequence of `pass1` calls and resets outside a step;
        `grid_state()` lags one step behind a single handle between steps (see `set_peer_three_call`)."""
        import torch.distributed as dist

        world, rank = dist.get_world_size(group), dist.get_rank(group)
        mine = (C.c_ubyte * _cabi.PEER_HANDLE_BYTES)()
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.as_peer_create(self.handle, world, rank, mine), "as_peer_create")
            on_gpu = dist.get_backend(group) == "nccl"
            t = torch.tensor(list(mine), dtype=torch.uint8, device=self.device if on_gpu else "cpu")
            gathered = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(gathered, t, group=group)
            blob = b"".join(bytes(g.cpu().tolist()) for g in gathered)
            _cabi.check(self.lib.as_peer_connect(self.handle, blob), "as_peer_connect")
        self._bind_global_stats()
        if three_call:
            self.set_peer_three_call(True)
        dist.barrier(group)  # nobody steps before every mapping exists
        return world, rank

    def connect_self(self, three_call: bool = False):
        """World of one (tests, single-GPU runs of a sharded script): the exchange kernel talks to itself."""
        mine = (C.c_ubyte * _cabi.PEER_HANDLE_BYTES)()
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.as_peer_create(self.handle, 1, 0, mine), "as_peer_create")
            _cabi.check(self.lib.as_peer_connect(self.handle, bytes(mine)), "as_peer_connect")
        self._bind_global_stats()
        if three_call:
            self.set_peer_three_call(True)

    def set_peer_three_call(self, enable: bool):
        """Global 3-call mode on connected peers (`as_peer_three_call`), switched between steps.  In it `step()` is
        refused, and this step's grid outcomes join the histograms -- summed over the shards -- at the exchange of
        the next `pass1`: between steps `grid_state()` / `grid_hist_tensor` lag one step behind one handle holding all
        envs, right after each `pass1` they are equal."""
        _cabi.check(self.lib.as_peer_three_call(self.handle, 1 if enable else 0), "as_peer_three_call")

    def _bind_global_stats(self):
        ptr = C.c_void_p()
        _cabi.check(self.lib.as_global_stats_device_ptr(self.handle, C.byref(ptr)), "as_global_stats_device_ptr")
        off = ptr.value - self.workspace.data_ptr()
        # device view of the step counters summed over all shards (int64 fields; see _cabi.AsStats)
        self.global_stats_tensor = self.workspace[off: off + C.sizeof(_cabi.AsStats)].view(torch.int64)
        self.global_exchange_tensor = self.workspace[off: off + C.sizeof(_cabi.AsExchange)].view(torch.int64)

    def peer_status(self) -> Dict[str, int]:
        world, rank, timeouts = C.c_int(), C.c_int(), C.c_int64()
        _cabi.check(self.lib.as_peer_status(self.handle, C.byref(world), C.byref(rank), C.byref(timeouts),
                                            self._stream()), "as_peer_status")
        return {"world": world.value, "rank": rank.value, "timeouts": timeouts.value}

    def fold_stats(self):
        """Between `step(..., finish=False)` and `finish_step(global)`: make this step's counters available in
        `stats_tensor` so they can be all-reduced over the shards first (promotion on the global mean)."""
        _cabi.check(self.lib.as_fold_stats(self.handle, self._stream()), "as_fold_stats")

    def all_reduce_exchange(self, buf: torch.Tensor, dist, group=None) -> torch.Tensor:
        """The plain-library route of a sharded step: `buf` (a copy of `exchange_tensor`, made after `fold_stats()`)
        summed over the ranks where it is additive -- the ten leading counters and, with the grid curriculum, the
        grid outcomes.  Hand the result to `finish_step`."""
        from .sharding import all_reduce_exchange

        return all_reduce_exchange(buf, bool(self.grid_bins), group)

    def finish_step(self, global_stats: Optional[torch.Tensor] = None):
        """Close the fused step: conditional no-reset fix-up, promotion rule (ENV:471-479), counters.  global_stats: a
        device tensor holding an AsExchange summed over the shards (see `all_reduce_exchange`)."""
        if global_stats is not None and global_stats.numel() * global_stats.element_size() < C.sizeof(_cabi.AsExchange):
            raise ValueError("global_stats must hold a whole AsExchange record (a copy of mdp.exchange_tensor)")
        _cabi.check(self.lib.as_finish_step(self.handle, _ptr(global_stats), self._stream()), "as_finish_step")

    # ------------------------------------------------------------------ 3-call path
    def pass1(self, views: PhysicsViews, actions: torch.Tensor, out: StepBuffers,
              episode_length: Optional[torch.Tensor] = None):
        self._check_views(views)
        _require(actions, torch.float32, self.device, "actions")
        stride = actions.stride(0) if self.num_envs > 1 else NUM_JOINTS
        if episode_length is not None:
            _require(episode_length, torch.int64, self.device, "episode_length")
        _cabi.check(self.lib.as_step_pass1(self.handle, C.byref(views.struct), actions.data_ptr(), stride,
                                           _ptr(episode_length), C.byref(out.step_out), self._stream()),
                    "as_step_pass1")

    def reset(self, env_origins: torch.Tensor, env_ids: Optional[torch.Tensor], out: StepBuffers,
              episode_length: Optional[torch.Tensor] = None):
        """`_reset_idx(env_ids)` minus the PhysX writes.  env_ids None: the envs the preceding `pass1` flagged, taken
        from the id list that pass compacted on the device -- no `.nonzero()`, no host round trip; `out.reset_ids[:n]`
        / `out.n_reset` (device) name them, rows are in that order.  With `regenerates`, the stones of the reset envs
        may have changed (grid curriculum: new bin and stones for every one of them): write them to the simulator too."""
        if env_ids is None:
            _cabi.check(self.lib.as_reset(self.handle, env_origins.data_ptr(), None, -1, _ptr(episode_length),
                                          C.byref(out.reset_out), self._stream()), "as_reset")
            self._keepalive = (env_origins,)
            return
        ids = env_ids.to(device=self.device, dtype=torch.int32).contiguous()
        _cabi.check(self.lib.as_reset(self.handle, env_origins.data_ptr(), ids.data_ptr(), ids.numel(),
                                      _ptr(episode_length), C.byref(out.reset_out), self._stream()), "as_reset")
        self._keepalive = (ids, env_origins)

    def pass2(self, views: PhysicsViews, out: StepBuffers):
        """ENV:567 after the PhysX writes of `_reset_idx`: makes `out.obs` final for a step in which envs reset."""
        self._check_views(views)
        _cabi.check(self.lib.as_step_pass2(self.handle, C.byref(views.struct), out.obs.data_ptr(), self._stream()),
                    "as_step_pass2")
        self._keepalive = (views, out)

    def no_reset(self):
        """The step's `reset_buf` was empty (DRL:360): no `_reset_idx`, no pass 2 -- makes the observations of `pass1`
        final.  Exactly one of `pass2` / `no_reset` closes every `pass1`; a no-op when none is open."""
        _cabi.check(self.lib.as_step_no_reset(self.handle, self._stream()), "as_step_no_reset")

    # ------------------------------------------------------------------ action path / symmetry
    def apply_action(self, actions: torch.Tensor, efforts: Optional[torch.Tensor] = None) -> torch.Tensor:
        _require(actions, torch.float32, self.device, "actions")
        if efforts is None:
            efforts = torch.empty(self.num_envs, NUM_JOINTS, dtype=torch.float32, device=self.device)
        stride = actions.stride(0) if self.num_envs > 1 else NUM_JOINTS
        _cabi.check(self.lib.as_apply_action(self.handle, actions.data_ptr(), stride, efforts.data_ptr(),
                                             self._stream()), "as_apply_action")
        return efforts

    def mirror_rows(self, rows: torch.Tensor, kind: str) -> torch.Tensor:
        """ENV:570-660: returns vstack((rows, mirrored(rows))). kind: 'obs' (dim 59) or 'actions' (dim 21)."""
        _require(rows, torch.float32, self.device, "rows")
        k = {"obs": 0, "actions": 1}[kind]
        dim = OBS_DIM if k == 0 else NUM_JOINTS
        if rows.dim() != 2 or rows.shape[1] != dim or not rows.is_contiguous():
            raise ValueError(f"rows must be contiguous (R,{dim})")
        out = torch.empty(2 * rows.shape[0], dim, dtype=torch.float32, device=self.device)
        _cabi.check(self.lib.as_mirror_rows(self.handle, rows.data_ptr(), out.data_ptr(), rows.shape[0], k,
                                            self._stream()), "as_mirror_rows")
        return out

    # ------------------------------------------------------------------ state in the reference's layouts
    _STATE_FIELDS = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "curriculum",
                     "potentials", "steps_pos", "steps_dphi")

    def export_state(self, fields: Optional[Tuple[str, ...]] = None) -> Dict[str, torch.Tensor]:
        """The MDP state in the reference's own buffers (ENV:48,74-78, DRL:179).  `fields`: only these (default all;
        `prev_target_index` / `next_target_index` come with `curr_target_index`) -- the S x 16-byte stone rows are the
        bulk of a full export, a caller that logs one counter per step should not pay for them."""
        N, S, dev = self.num_envs, self.num_steps, self.device
        want = set(self._STATE_FIELDS if fields is None else fields)
        if want & {"prev_target_index", "next_target_index"}:
            want.add("curr_target_index")
        unknown = want - set(self._STATE_FIELDS) - {"prev_target_index", "next_target_index"}
        if unknown:
            raise KeyError(f"unknown state fields: {sorted(unknown)}")
        shapes = {"potentials": ((N,), torch.float32), "steps_pos": ((N, S, 3), torch.float32),
                  "steps_dphi": ((N, S), torch.float32)}
        d = {k: torch.empty(*shapes.get(k, ((N,), torch.int64))[0], dtype=shapes.get(k, ((N,), torch.int64))[1], device=dev)
             for k in self._STATE_FIELDS if k in want}
        st = _cabi.AsMdpState(*[_ptr(d.get(k)) for k in self._STATE_FIELDS])
        _cabi.check(self.lib.as_export_state(self.handle, C.byref(st), self._stream()), "as_export_state")
        if "curr_target_index" in d:
            d["prev_target_index"] = torch.clamp(d["curr_target_index"] - 1, 0, S - 1)  # ENV:76
            d["next_target_index"] = torch.clamp(d["curr_target_index"] + 1, 0, S - 1)  # ENV:77
        return d

    def export_stone_poses(self, env_ids: Optional[torch.Tensor] = None, view_poses: Optional[torch.Tensor] = None):
        """Stone poses of `env_ids` (None: all envs) the way PhysX takes them: rows of the object-major
        (S*N,7) x,y,z,w tensor plus their view indices -- `steps.root_physx_view.set_transforms(view_poses,
        indices=view_ids)` replaces ENV:119-120 + rigid_object_collection.py:295-301 (no whole-tensor clone, quaternion
        conversion or transpose).  `view_poses` may be a persistent buffer; rows of other envs are left untouched."""
        N, S, dev = self.num_envs, self.num_steps, self.device
        if view_poses is None:
            view_poses = torch.zeros(S * N, 7, dtype=torch.float32, device=dev)
        _require(view_poses, torch.float32, dev, "view_poses")
        if tuple(view_poses.shape) != (S * N, 7) or not view_poses.is_contiguous():
            raise ValueError("view_poses must be a contiguous (S*N,7) tensor")
        ids_ptr, k = None, N
        if env_ids is not None:
            env_ids = env_ids.to(device=dev, dtype=torch.int32).contiguous()
            ids_ptr, k = env_ids.data_ptr(), env_ids.numel()
        view_ids = torch.empty(S * k, dtype=torch.int32, device=dev)
        if k:
            _cabi.check(self.lib.as_export_stone_poses(self.handle, ids_ptr, k, view_poses.data_ptr(),
                                                       view_ids.data_ptr(), self._stream()), "as_export_stone_poses")
        self._keepalive_poses = (env_ids, view_poses, view_ids)
        return view_poses, view_ids

    def import_state(self, state: Dict[str, torch.Tensor]):
        keep = {}

        def get(name, dtype, shape):
            t = state.get(name)
            if t is None:
                return None
            t = t.to(device=self.device, dtype=dtype).contiguous()
            if tuple(t.shape) != shape:
                raise ValueError(f"{name}: expected shape {shape}, got {tuple(t.shape)}")
            keep[name] = t
            return t.data_ptr()

        N, S = self.num_envs, self.num_steps
        st = _cabi.AsMdpState(
            get("curr_target_index", torch.int64, (N,)), get("swing_leg", torch.int64, (N,)),
            get("target_reach_count", torch.int64, (N,)), get("episode_length_buf", torch.int64, (N,)),
            get("curriculum", torch.int64, (N,)), get("potentials", torch.float32, (N,)),
            get("steps_pos", torch.float32, (N, S, 3)), get("steps_dphi", torch.float32, (N, S)))
        _cabi.check(self.lib.as_import_state(self.handle, C.byref(st), self._stream()), "as_import_state")
        self._keepalive = keep

    # ------------------------------------------------------------------ grid curriculum extension
    def grid_state(self):
        """(bins (N,) uint8, attempts (B*B,) int64, successes (B*B,) int64) of the difficulty-grid curriculum."""
        bins = torch.empty(self.num_envs, dtype=torch.uint8, device=self.device)
        hist = torch.empty(512, dtype=torch.int32, device=self.device)
        _cabi.check(self.lib.as_grid_state(self.handle, bins.data_ptr(), None, hist.data_ptr(), None,
                                           self._stream()), "as_grid_state")
        nb = self.grid_bins * self.grid_bins
        # (uint32 counters: widen, then drop the sign extension)
        return bins, hist[:nb].long() & 0xFFFFFFFF, hist[256:256 + nb].long() & 0xFFFFFFFF

    def set_grid_state(self, bins: Optional[torch.Tensor] = None, attempts=None, successes=None):
        """bins (N,) with values < B*B; attempts and successes (B*B,) each, 0 <= successes <= attempts < 2^32 (the
        precondition of oracle/grid_curriculum.py).  Anything else raises ValueError before the handle is touched."""
        nb = self.grid_bins * self.grid_bins
        b = None
        if bins is not None:
            b64 = torch.as_tensor(bins).detach().to("cpu", torch.int64)
            if tuple(b64.shape) != (self.num_envs,):
                raise ValueError(f"bins must have shape ({self.num_envs},), got {tuple(b64.shape)}")
            if b64.numel() and (int(b64.min()) < 0 or int(b64.max()) >= nb):
                raise ValueError(f"bins must lie in [0, {nb}) for a {self.grid_bins}x{self.grid_bins} grid")
            b = b64.to(device=self.device, dtype=torch.uint8)
        hist = None
        if (attempts is None) != (successes is None):
            raise ValueError("attempts and successes are set together")
        if attempts is not None:
            att = torch.as_tensor(attempts).detach().to("cpu", torch.int64)
            succ = torch.as_tensor(successes).detach().to("cpu", torch.int64)
            for name, x in (("attempts", att), ("successes", succ)):
                if tuple(x.shape) != (nb,):
                    raise ValueError(f"{name} must have shape ({nb},), got {tuple(x.shape)}")
                if nb and (int(x.min()) < 0 or int(x.max()) > 0xFFFFFFFF):
                    raise ValueError(f"{name} must lie in [0, 2^32): the histogram counters are uint32")
            if bool((succ > att).any()):
                raise ValueError("successes must not exceed attempts in any bin")
            h = torch.zeros(512, dtype=torch.int64)
            h[:nb] = att
            h[256:256 + nb] = succ
            hist = torch.where(h > 0x7FFFFFFF, h - (1 << 32), h).to(device=self.device, dtype=torch.int32)  # uint32 bits
        _cabi.check(self.lib.as_grid_state(self.handle, None, _ptr(b), None, _ptr(hist), self._stream()),
                    "as_grid_state")
        self._keepalive = (b, hist)

    # ------------------------------------------------------------------ exact checkpoint / resume (SURVEY section 5)
    def snapshot(self, include_stones: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Opaque device blob of the whole MDP state: packed state words, stone windows (and rows), grid bins and
        histograms, pending promotion, Philox step counter.  Stream-ordered, no synchronisation."""
        n = int(self.lib.as_snapshot_bytes(self.handle, 1 if include_stones else 0))
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
        if out.numel() != n or out.dtype != torch.uint8 or out.device != self.device or not out.is_contiguous():
            raise ValueError(f"snapshot buffer must be a contiguous uint8 tensor of {n} bytes on {self.device}")
        _cabi.check(self.lib.as_snapshot(self.handle, out.data_ptr(), 1 if include_stones else 0, self._stream()),
                    "as_snapshot")
        return out

    def restore(self, blob: torch.Tensor, include_stones: bool = True):
        """Put a `snapshot()` back (same num_envs; `include_stones` as it was taken)."""
        n = int(self.lib.as_snapshot_bytes(self.handle, 1 if include_stones else 0))
        if blob.numel() != n or blob.dtype != torch.uint8:
            raise ValueError(f"snapshot of {blob.numel()} bytes does not fit this handle ({n} bytes expected)")
        blob = blob.to(self.device).contiguous()
        _cabi.check(self.lib.as_restore(self.handle, blob.data_ptr(), 1 if include_stones else 0, self._stream()),
                    "as_restore")
        self._keepalive = blob

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """Checkpoint for an exact resume: `snapshot` is what `load_state_dict` restores (it holds the Philox position,
        the pending promotion and the grid-curriculum state too); the reference-layout buffers of `export_state()` ride
        along for inspection."""
        d = {k: v.cpu() for k, v in self.export_state().items()}
        d["snapshot"] = self.snapshot(include_stones=True).cpu()
        d["meta"] = torch.tensor([_cabi.ABI_VERSION, self.num_envs, self.env_id_offset, self.seed,
                                  int(self.params.flags), self.grid_bins, self.num_steps], dtype=torch.int64)
        return d

    def load_state_dict(self, d: Dict[str, torch.Tensor]):
        meta = [int(x) for x in d["meta"].tolist()]
        mine = [_cabi.ABI_VERSION, self.num_envs, self.env_id_offset, self.seed, int(self.params.flags), self.grid_bins,
                self.num_steps]
        names = ["abi", "num_envs", "env_id_offset", "seed", "flags", "grid_bins", "num_steps"]
        for name, a, b in zip(names, meta, mine):
            if a != b:
                raise ValueError(f"checkpoint was taken with {name}={a}, this handle has {name}={b}")
        self.restore(d["snapshot"], include_stones=True)

    def read_stats(self) -> Dict[str, float]:
        s = _cabi.AsStats()
        _cabi.check(self.lib.as_read_stats(self.handle, C.byref(s), self._stream()), "as_read_stats")
        return s.as_dict()
