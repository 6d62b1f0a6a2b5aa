/*
 * allsteps_b200.h -- C ABI of the B200-native Allsteps-v0 batched MDP step.
 *
 * The reference (xindonglin99/allsteps_isaaclab) has no FFI layer: the path is six Python hook methods of
 * `AllstepsEnv(DirectRLEnv)`.  This header is the boundary a maintainer binds instead (ctypes stub in
 * INTEGRATION.md; allsteps_isaaclab_b200/_cabi.py is that stub).  Every entry point names the reference code
 * it replaces:  ENV = source/isaaclab_tasks/isaaclab_tasks/direct/allsteps/allsteps_env.py,
 *               DRL = source/isaaclab/isaaclab/envs/direct_rl_env.py,  CFG = .../allsteps/allsteps_env_cfg.py.
 *
 * Conventions
 *  - plain C: pointers, sizes, POD structs.  No torch / CUDA types; a stream is passed as `void*`
 *    (a `cudaStream_t`, e.g. `torch.cuda.current_stream().cuda_stream`).
 *  - every pointer inside AsStateIn / AsStepOut / AsResetOut is a DEVICE pointer owned by the caller.
 *  - the library never allocates device memory and never synchronises the stream or the device on the step path
 *    (only the *_export_* / as_read_stats helpers, which return host data, synchronise the given stream).
 *  - return value: 0 on success, negative AS_ERR_* otherwise; text via as_last_error() (thread local).
 *  - built only for sm_100a.  There is no CPU fallback: on a machine without a usable device every compute
 *    entry point returns AS_ERR_CUDA.
 */
#ifndef ALLSTEPS_B200_H_
#define ALLSTEPS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AS_ABI_VERSION 5

#define AS_NUM_JOINTS 21  /* CFG:57  action_space            */
#define AS_NUM_STONES 20  /* CFG:90  num_steps: the default course length (AsParams.num_steps = 0) */
#define AS_MIN_STONES 3   /* stones 0..2 are the fixed start stones, ENV:144-150 */
#define AS_MAX_STONES 32  /* the packed state word holds curr_target_index in 5 bits */
#define AS_OBS_DIM 59     /* CFG:58  observation_space       */
#define AS_NUM_LEVELS 10  /* ENV:45  max_curriculum + 1      */
#define AS_ROOT_STATE_DIM 13
#define AS_NUM_REWARD_TERMS 10
#define AS_TILE_ENVS 128  /* envs handled by one CTA; sharded slices should start on a multiple of 4 envs */

enum {
  AS_OK = 0,
  AS_ERR_INVALID = -1, /* bad argument (null pointer, bad size, unsupported stride ...) */
  AS_ERR_CUDA = -2,    /* a CUDA runtime call failed; as_last_error() has the CUDA message  */
  AS_ERR_STATE = -3,   /* call sequence violated (e.g. a fused step left open)             */
  AS_ERR_PEER = -4     /* a peer exchange timed out earlier: sticky, the shards may have diverged */
};

/* AsParams.flags */
enum {
  AS_FLAG_INTENDED_REGEN = 1u << 0, /* extension: regenerate stones of a reset env whose index had passed
                                       num_steps/2 BEFORE the index reset.  Off = reference-exact: the test at
                                       ENV:497 runs after ENV:492 and is never true (SURVEY D3).            */
  AS_FLAG_SKIP_PASS2 = 1u << 1,     /* extension: never run the second `_compute_useful_values` pass
                                       (ENV:567, SURVEY D7) for envs that did not reset.  Off = reference. */
  AS_FLAG_GRID_CURRICULUM = 1u << 2,/* extension: pitch x yaw difficulty grid sampling at regeneration:
                                       every env that resets -- in as_step_fused or in as_reset -- gets a new
                                       bin and new stones (see as_grid_state).                              */
  AS_FLAG_MISSED_STEP = 1u << 3     /* extension (BASELINE north_star "missed-step termination"; the reference's
                                       ENV:396-405 has none, SURVEY D4): an env also terminates when its swing foot
                                       has come down below the top of the stone it is heading for, outside that stone's
                                       footprint -- swing_foot_z < stone_z + missed_step_height  and
                                       |swing_foot_xy - stone_xy| >= step_radius, swing leg and current stone taken as
                                       they are BEFORE the pass updates them.  Specification: AllstepsOracle(
                                       missed_step_height=...) in oracle/allsteps_oracle.py.  Off = reference.  */
};

/* Constants of the task: CFG:52-235 plus the values hard-coded in ENV:41-59.  Tables that the reference builds
 * with torch (linspace) are filled in by the host with torch so that they are bit-identical. */
typedef struct AsParams {
  float step_dt;                   /* sim.dt * decimation, DRL step_dt                                  */
  int32_t max_episode_length;      /* DRL:248-250 -> 900                                                */
  float step_radius;               /* CFG:97                                                            */
  float dist_lower;                /* ENV:41 dist_range[0]                                              */
  float dist_upper[AS_NUM_LEVELS]; /* linspace(dist_range, 10), ENV:129                                 */
  float yaw_range_deg[2];          /* ENV:43                                                            */
  float pitch_range_deg[2];        /* ENV:42                                                            */
  float init_step_separation;      /* ENV:50                                                            */
  int32_t max_level;               /* ENV:45                                                            */
  float termination_height[AS_NUM_LEVELS]; /* linspace(0.75, 0.45, 10), ENV:46                          */
  float applied_gain[AS_NUM_LEVELS];       /* linspace(1.2, 1.2, 10),  ENV:47                           */
  float progress_threshold;        /* ENV:53 (12)                                                       */
  float contact_epsilon;           /* ENV:32                                                            */
  int32_t stop_frames;             /* ENV:56 (<= 3)                                                     */
  float energy_cost_scale, actions_cost_scale, alive_reward_scale, dof_vel_scale;   /* CFG:222-225      */
  float joint_at_limit_cost_scale, death_cost;                                      /* CFG:226-227      */
  float termination_height_absolute; /* CFG:228                                                         */
  float max_root_speed;            /* ENV:402 (5.0)                                                     */
  float noise_span, noise_lower;   /* (hi - lo) and lo of CFG:232, as MATH:1331 evaluates them          */
  float clip_lower, clip_upper;    /* CFG:233                                                           */
  float default_root_pos[3];       /* walker3d.py:36                                                    */
  float joint_lower[AS_NUM_JOINTS], joint_upper[AS_NUM_JOINTS]; /* robot.data.joint_pos_limits[0]       */
  float joint_gears[AS_NUM_JOINTS];/* CFG:133-155                                                       */
  float reset_pose[AS_NUM_JOINTS]; /* ENV:505-511                                                       */
  int32_t mirror_src[AS_NUM_JOINTS]; /* ENV:522-526: joint j takes the value of joint mirror_src[j] ... */
  float mirror_sign[AS_NUM_JOINTS];  /* ... times mirror_sign[j]                                        */
  float missed_step_height;        /* AS_FLAG_MISSED_STEP: metres above the stone's position below which the swing
                                      foot's body origin counts as "down" (extension, no reference counterpart) */
  uint32_t flags;
  uint32_t grid_bins;              /* AS_FLAG_GRID_CURRICULUM: bins per axis (<= 16), else 0            */
  uint32_t num_steps;              /* CFG:90: stones per course, S, in AS_MIN_STONES..AS_MAX_STONES; 0 = AS_NUM_STONES.
                                      Every "S" below is this value of the handle.                      */
  uint64_t seed;                   /* Philox key                                                        */
} AsParams;

/* Device views of what PhysX publishes after `scene.update` (DRL:347).  Row strides are in ELEMENTS (floats);
 * a stride equal to the row width with a 16-byte aligned base takes the TMA-staged fast path, anything else
 * (e.g. the (N,13) `root_state_w` views Isaac Lab hands out) takes the strided path. */
typedef struct AsStateIn {
  const float* root_pos;      int64_t root_pos_stride;     /* robot.data.root_pos_w      (N,3)              */
  const float* root_quat;     int64_t root_quat_stride;    /* robot.data.root_quat_w     (N,4) w,x,y,z      */
  const float* root_lin_vel;  int64_t root_lin_vel_stride; /* robot.data.root_lin_vel_w  (N,3)              */
  const float* body_pos;      int64_t body_env_stride;     /* robot.data.body_pos_w      (N,B,3)            */
  int64_t body_row_stride;                                  /* floats between bodies of one env (3 or 13)    */
  int32_t right_foot_row, left_foot_row, torso_row;         /* ENV:87-88                                     */
  int32_t quat_xyzw;  /* 1: root_quat is x,y,z,w as PhysX' own root transforms are (skips Isaac Lab's convert_quat,
                         articulation_data.py:372-379); 0: w,x,y,z as robot.data.root_quat_w                        */
  const float* joint_pos;     int64_t joint_pos_stride;    /* robot.data.joint_pos       (N,21)             */
  const float* joint_vel;     int64_t joint_vel_stride;    /* robot.data.joint_vel       (N,21)             */
  const float* contact_right; int64_t contact_right_stride;/* sensor_right.data.force_matrix_w (N,1,S,3),   */
  const float* contact_left;  int64_t contact_left_stride; /* sensor_left.data.force_matrix_w  (N,1,S,3),   */
                                                            /* S = AsParams.num_steps; strides >= 3 S         */
  const float* env_origins;                                 /* scene.env_origins (N,3) contiguous            */
} AsStateIn;

/* Results of one step, the tuple DRL:383 returns.  `terminated` / `time_out` are 1-byte 0/1 (torch.bool). */
typedef struct AsStepOut {
  float* obs;            /* (N,59)  ENV:326-345                                                            */
  float* reward;         /* (N)     ENV:347-394                                                            */
  uint8_t* terminated;   /* (N)     ENV:405 fell | so_fast | died                                          */
  uint8_t* time_out;     /* (N)     ENV:399                                                                */
  float* reward_terms;   /* optional (N,10): alive, progress, roll, pitch, speed, energy, action, limit,
                            step, bonus (costs positive) -- for per-term manager logging; NULL to skip     */
  uint8_t* dones;        /* optional (N): terminated | time_out, what RlGamesVecEnvWrapper.step hands to
                            rl_games (isaaclab_rl/rl_games.py:256) and DirectRLEnv keeps as reset_buf      */
  float obs_clip;        /* > 0: obs is written as clamp(obs, -obs_clip, +obs_clip), the `clip_obs` step of
                            RlGamesVecEnvWrapper._process_obs (isaaclab_rl/rl_games.py:293; NaN is kept, like
                            torch.clamp), so the wrapper can hand the buffer on as it is.  0: raw (ENV:326-345).
                            as_step_pass2 applies the value given to the as_step_pass1 before it.           */
  uint32_t flags;        /* AS_STEP_* bits                                                                 */
  float* final_obs;      /* optional (N,59), 4-byte aligned, not overlapping obs; NULL to skip.  The final
                            observation of every env that resets in this step (terminated | time_out): the row the
                            reference's `_get_observations()` (ENV:326-345) returns when called between `_get_dones` /
                            `_get_rewards` and `_reset_idx` -- h, roll, pitch, v_b, scaled joint positions and clipped
                            joint velocities of the step's physics input, foot_contact and targets_b as pass 1 left
                            them -- clamped by obs_clip like obs.  What `V(s_T)` of a truncated episode needs, since
                            `obs` holds the start pose of an env that reset.  Written at the env's own row, only for the
                            envs that reset; other rows, and the whole buffer in a step in which no env resets, are
                            left untouched.  Honoured by as_step_fused and as_step_pass1 (the envs pass 1 flagged,
                            whatever ids as_reset is given later); the generic kernel instantiation runs when set. */
} AsStepOut;
/* AsStepOut.flags */
enum {
  AS_STEP_DEFER_FINISH = 1u << 0  /* as_step_fused: the caller is going to call as_fold_stats and hand the summed
                                     statistics to as_finish_step(global_stats) -- the step kernel must leave the step
                                     open (by default its last CTA closes the step itself and as_finish_step only
                                     checks a flag) */
};

/* What `_reset_idx` hands to PhysX (ENV:563-565).  Rows are written AT THE ENV'S OWN ROW (full-size buffers),
 * only for envs that reset; `reset_ids[0 .. *n_reset)` lists them (unordered).  All optional. */
typedef struct AsResetOut {
  float* root_state;     /* (N,13) pos, quat wxyz, lin vel, ang vel                                        */
  float* joint_pos;      /* (N,21)                                                                         */
  float* joint_vel;      /* (N,21)                                                                         */
  int32_t* reset_ids;    /* (N)                                                                            */
  int32_t* n_reset;      /* (1)                                                                            */
} AsResetOut;

/* Step statistics, accumulated on the device and summed over ranks by the caller (NCCL) when sharded. */
typedef struct AsStats {
  int64_t n_envs;        /* envs that contributed                                                          */
  int64_t n_reset, n_terminated, n_time_out, n_fell, n_so_fast, n_died;
  int64_t n_advanced;    /* stones reached (index advances) in this step, both passes.  3-call path: pass 1
                            counts the pass-2 advances it speculates; as_step_no_reset, or as_step_pass2
                            finding the device-side list empty, takes them back with pass 2              */
  int64_t sum_target_index; /* sum of curr_target_index after pass 1: numerator of ENV:471                 */
  int64_t n_regenerated;
  int64_t level;         /* current curriculum level (max over envs when per-env levels are in use)        */
  int64_t step_counter;
  double sum_reward;
  int64_t n_missed;      /* AS_FLAG_MISSED_STEP: envs terminated by a missed step (this shard)             */
} AsStats;

/* What the shards of a sharded run exchange per step: the step statistics (only the leading AS_NUM_ADDITIVE_STATS
 * int64 fields are summed) followed by this step's difficulty-grid outcomes (AS_FLAG_GRID_CURRICULUM: episodes ended
 * per bin, and how many of them had passed half of the stones; zero otherwise).  One contiguous device record, so that
 * the plain-library route is one all-reduce over a byte range. */
#define AS_NUM_ADDITIVE_STATS 10
#define AS_MAX_GRID_CELLS 256
typedef struct AsExchange {
  AsStats stats;
  uint32_t grid_attempts[AS_MAX_GRID_CELLS];
  uint32_t grid_successes[AS_MAX_GRID_CELLS];
} AsExchange;

typedef struct AsHandle AsHandle;

/* ---- lifetime --------------------------------------------------------------------------------------- */
int as_abi_version(void);
const char* as_last_error(void);
/* Bytes of device workspace needed for `num_envs` envs (MDP state: stones, packed state, control block) with courses
 * of AS_NUM_STONES stones. */
int64_t as_workspace_bytes(int64_t num_envs);
/* The same for the course length of `params` (params->num_steps); 0 when num_envs <= 0 or num_steps is out of range. */
int64_t as_workspace_bytes_for(const AsParams* params, int64_t num_envs);
/* `workspace`: device memory of as_workspace_bytes_for(params, num_envs) bytes, 256-byte aligned, zero-initialised by this call.
 * `env_id_offset`: global id of local env 0 (env-id sharding; Philox is keyed by global id).
 * Replaces AllstepsEnv.__init__ buffer allocation, ENV:41-96. */
int as_create(const AsParams* params, int64_t num_envs, int64_t env_id_offset, int device,
              void* workspace, int64_t workspace_bytes, void* stream, AsHandle** out);
void as_destroy(AsHandle* h);

/* ---- stones: ENV:106-174 `_generate_foot_steps` -------------------------------------------------------
 * env_ids: NULL = all envs, else `n_ids` local ids (device, int32).  uniforms: NULL = in-kernel Philox at the
 * current step counter, else device (5,N,S) floats indexed by LOCAL env id (replay of external draws); S is
 * AsParams.num_steps.
 * levels are taken from the per-env state. */
int as_generate_stones(AsHandle* h, const float* env_origins, const int32_t* env_ids, int64_t n_ids,
                       const float* uniforms, void* stream);

/* ---- the fused step: DRL:351-375 in one launch (+ a device-side conditional fix-up launch) -------------
 * episode counter += 1, pass 1 (ENV:276-324), dones (ENV:396-405), rewards (ENV:347-394), masked reset
 * (ENV:469-565), pass 2 (ENV:567) and observations (ENV:326-345).  `actions` (N,21) raw policy output, clamped
 * to [-1,1] inside (ENV:267-268).  For envs that reset, pass 2 sees the root / joint rows this call generates,
 * zero contacts and unchanged body positions (what `robot.data` holds between the PhysX writes and the next
 * physics step). */
int as_step_fused(AsHandle* h, const AsStateIn* in, const float* actions, int64_t actions_stride,
                  const AsStepOut* out, const AsResetOut* reset_out, void* stream);

/* ---- the same step as three calls, for hosts that run PhysX between them --------------------------------
 * pass1:  `_get_dones` + `_get_rewards`; `obs` is final only after as_step_pass2 or as_step_no_reset (below).
 *         episode_length: optional device int64 (N) owned by DirectRLEnv (already incremented, DRL:351);
 *         NULL = the library keeps and increments its own counter.
 * reset:  `_reset_idx(env_ids)` minus the PhysX writes: promotion rule, MDP state reset, start pose rows.
 *         Compact outputs: row i of the AsResetOut buffers belongs to env_ids[i].
 *         env_ids == NULL with n_ids < 0: "the envs as_step_pass1 just flagged" -- the id list that pass compacted on
 *         the device (no `.nonzero()` / host round trip as in DRL:359); rows come out in list order, `reset_ids` and
 *         `n_reset` of AsResetOut say which and how many; when the list is empty the as_step_pass2 that follows acts
 *         as as_step_no_reset.
 *         Called without a preceding as_step_pass1 (DirectRLEnv.reset() runs `_reset_idx(all ids)` before the first
 *         step, DRL:256-279) it evaluates the promotion rule on the indices as they are and advances the Philox
 *         step counter itself.
 *         With AS_FLAG_GRID_CURRICULUM or AS_FLAG_INTENDED_REGEN it regenerates stones by the rule of the fused step
 *         (every listed env with the grid, those past num_steps/2 with intended regeneration; AsStats.n_regenerated
 *         counts them): the caller writes the stones of the reset envs to its simulator (as_export_state /
 *         as_export_stone_poses).  Grid outcomes: see as_grid_state.
 * pass2:  the second `_compute_useful_values` over ALL envs + `_get_observations`, on the post-write state.  No
 *         call-order precondition (ENV:567 runs whether or not a pass preceded the reset). */
int as_step_pass1(AsHandle* h, const AsStateIn* in, const float* actions, int64_t actions_stride,
                  const int64_t* episode_length, const AsStepOut* out, void* stream);
int as_reset(AsHandle* h, const float* env_origins, const int32_t* env_ids, int64_t n_ids,
             int64_t* episode_length, const AsResetOut* compact_out, void* stream);
int as_step_pass2(AsHandle* h, const AsStateIn* in, float* obs, void* stream);
/* DRL:360 found no env to reset, so `_reset_idx` -- and with it pass 2 -- does not run this step: the observations of
 * as_step_pass1 are made final.  (as_step_pass1 works like the fused step: it ASSUMES that some env resets, runs pass 2
 * for every env that does not on the spot -- their physics cannot change between DRL:354 and ENV:567 -- and leaves the
 * result in the second state buffer and in `obs`; as_step_pass2 then only redoes the envs that did reset, from the views
 * as they are after the PhysX writes, and switches buffers.  This call takes the assumption back: observation columns
 * 48..58 as pass 1 left them, state of pass 1.)  Call it, or as_reset + as_step_pass2, once per as_step_pass1; a no-op
 * when no pass 1 is open. */
int as_step_no_reset(AsHandle* h, void* stream);

/* ---- curriculum: ENV:470-479 -----------------------------------------------------------------------------
 * The step kernels leave per-step statistics in the control block; as_finish_step folds them, applies the
 * promotion rule (mean(curr_target_index) > 12 and at least one reset => level+1) for the NEXT step and clears
 * the accumulators.  When envs are sharded, pass `global` = a device AsExchange summed over ranks (NCCL: the first
 * AS_NUM_ADDITIVE_STATS int64 of `stats` and, with AS_FLAG_GRID_CURRICULUM, the two grid arrays) to promote on the
 * global mean and to keep every shard's difficulty-grid histograms equal to those of one handle holding all envs;
 * NULL = this shard's own envs (what `--distributed` replicas do). */
int as_stats_device_ptr(AsHandle* h, AsStats** device_stats);  /* = the head of the record as_exchange_device_ptr gives */
/* This shard's exchange record (`local`: statistics folded by as_fold_stats / the finish kernel + this step's grid
 * outcomes) and the record summed over all shards by the peer-memory exchange (`global`; after as_peer_connect). */
int as_exchange_device_ptr(AsHandle* h, AsExchange** local, AsExchange** global);
/* Optional, between as_step_fused and as_finish_step: fold this step's counters into the device AsStats now, so
 * that the caller can all-reduce them and pass the sum to as_finish_step(global_stats) for a promotion decision on
 * the global mean in the same step. */
int as_fold_stats(AsHandle* h, void* stream);
/* Closes the step opened by as_step_fused (required once per fused step, on the same stream; the buffers given
 * to as_step_fused must stay alive until then because the conditional no-reset fix-up re-reads them). */
int as_finish_step(AsHandle* h, const AsExchange* global, void* stream);
int as_read_stats(AsHandle* h, AsStats* host_out, void* stream); /* synchronises `stream` */

/* ---- the promotion rule's cross-shard sum over NVLink peer memory (SURVEY 8(e): the ONE cross-env dependency of the
 * path, `mean(curr_target_index) > 12` over ALL envs, ENV:471) --------------------------------------------------
 * One process per GPU.  as_peer_create allocates this shard's 4-KB exchange buffer and returns its CUDA IPC handle
 * (AS_PEER_HANDLE_BYTES bytes); the caller gathers the handles of all ranks (any transport, e.g.
 * torch.distributed.all_gather) and hands them, in rank order, to as_peer_connect.  From then on the last CTA of the
 * fused step kernel folds this shard's step counters, stores them into every peer's buffer through NVLink, waits for
 * the peers' stores of the same step, sums them and closes the step on that global sum (as_finish_step(h, NULL,
 * stream) is left with a step in which no env of any shard reset).  When the step kernel leaves the step open
 * (AS_STEP_DEFER_FINISH, or the regeneration kernels behind it), as_finish_step(h, NULL, stream) launches ONE small
 * kernel for the fold and the exchange, followed by the finish kernel deciding on the sum.  Either way this is the
 * fused replacement of as_fold_stats + NCCL all-reduce + as_finish_step(global).  Every rank must call as_step_fused /
 * as_finish_step the same number of times.  A peer that does not deliver within ALLSTEPS_PEER_TIMEOUT_MS (default
 * 10 s; 0 = no limit) is counted in `*timeouts` of as_peer_status; the step closes on this shard's own record (a partial
 * sum is never used) and every later step is refused with the sticky AS_ERR_PEER (no hang).  world == 1 is allowed
 * (self-exchange).  as_global_stats_device_ptr: the summed AsStats (first 10 fields; the rest is this shard's). */
#define AS_PEER_HANDLE_BYTES 64
#define AS_MAX_PEERS 16
int as_peer_create(AsHandle* h, int world, int rank, void* ipc_handle_out);
int as_peer_connect(AsHandle* h, const void* ipc_handles_in_rank_order);
int as_peer_status(AsHandle* h, int* world, int* rank, int64_t* timeouts, void* stream); /* synchronises `stream` */
int as_global_stats_device_ptr(AsHandle* h, AsStats** device_stats);
/* Global 3-call mode (enable != 0; 0 switches it off again, between steps).  Valid after as_peer_connect, otherwise
 * AS_ERR_STATE; also AS_ERR_STATE while a step is open.  With it, a sharded run through the 3-call path (as_step_pass1
 * -> as_reset -> as_step_pass2 / as_step_no_reset) is bit-identical to one handle holding all envs: outputs, state,
 * levels, grid bins and stones.  as_step_pass1 launches one exchange behind pass 1 that sums the flagged count and the
 * indices over the shards and there decides the promotion of ENV:471 and "did any env reset" (DRL:359-360): when an env
 * of ANY shard reset, as_step_no_reset -- and as_step_pass2 on an empty device-side list -- keep pass 2 for every env
 * of this shard, as the reference does, instead of taking it back; as_reset uses the exchanged promotion.  A reset
 * outside a step (no as_step_pass1 open) exchanges too, right before it resets.  So every rank must make the same
 * sequence of as_step_pass1 / reset-outside-a-step calls (a reset outside a step with a non-empty id list); a rank that
 * does not meets the sticky AS_ERR_PEER of the exchange's time limit, not a hang.  Grid histograms: see as_grid_state.
 * Resets the caller adds that pass 1 did not flag (extra termination terms) reset correctly on their own shard but do
 * not count toward the global any-reset and promotion tests.  as_step_fused on a handle in this mode: AS_ERR_STATE. */
int as_peer_three_call(AsHandle* h, int32_t enable);

/* ---- action path: ENV:257-274 `_pre_physics_step` + `_apply_action` --------------------------------------
 * efforts[n,j] = applied_gain[level[n]] * joint_gears[j] * clamp(actions[n,j], -1, 1)
 * Any row stride >= 21 and any 4-byte aligned address is accepted; dense rows (stride 21) with `actions` and `efforts`
 * on 16-byte boundaries take the bulk-copy path (full 128-env tiles through shared memory), everything else an element
 * loop with the same results.  Isaac Lab calls `_apply_action` `decimation` times per env step with unchanged inputs:
 * one call per env step is enough (INTEGRATION.md). */
int as_apply_action(AsHandle* h, const float* actions, int64_t actions_stride, float* efforts, void* stream);

/* ---- mirror-symmetry augmentation: ENV:570-660 `get_symmetric_states_*` ----------------------------------
 * out (2*rows, dim): rows [0,rows) = copy of `in`, rows [rows, 2*rows) = mirrored.  kind: 0 = observations
 * (dim 59), 1 = actions / mus (dim 21).  `in` and `out` on 16-byte boundaries and a row count that is a multiple of 4
 * take the bulk-copy path (128-row tiles through shared memory: every element read once, written twice); other
 * shapes / alignments an element loop with the same results. */
int as_mirror_rows(AsHandle* h, const float* in, float* out, int64_t rows, int32_t kind, void* stream);
/* The same for up to four tensors in ONE launch -- what A2CAgentSymmetry.play_steps does to `obses`, `actions` and
 * `mus` every PPO epoch (learning/a2c_ppo_mirroring.py:32-38 -> get_symmetric_states_rl_games, ENV:611-660). */
typedef struct AsMirrorJob {
  const float* in;   /* (rows, dim)                                             */
  float* out;        /* (2*rows, dim): rows [0,rows) copy, [rows,2*rows) mirror */
  int64_t rows;
  int32_t kind;      /* 0 observations (dim 59), 1 actions / mus (dim 21)       */
  int32_t _pad;
} AsMirrorJob;
int as_mirror_batch(AsHandle* h, const AsMirrorJob* jobs, int32_t n_jobs, void* stream);

/* ---- state exchange in the reference's own layouts (checkpoint / replay / tests) -------------------------
 * All pointers device, optional (NULL = skip).  int64 arrays as in ENV:48,74-78 and DRL:179. */
typedef struct AsMdpState {
  int64_t* curr_target_index; /* (N) */
  int64_t* swing_leg;         /* (N) */
  int64_t* target_reach_count;/* (N) */
  int64_t* episode_length;    /* (N) */
  int64_t* curriculum;        /* (N) */
  float* potentials;          /* (N) */
  float* steps_pos;           /* (N,S,3), S = AsParams.num_steps */
  float* steps_dphi;          /* (N,S)   */
} AsMdpState;
int as_export_state(AsHandle* h, const AsMdpState* dst, void* stream);
int as_import_state(AsHandle* h, const AsMdpState* src, void* stream);

/* ---- exact checkpoint / resume (SURVEY section 5) -----------------------------------------------------------
 * A snapshot is one opaque device blob: control block (state parity, pending promotion, Philox step counter, folded
 * statistics, difficulty-grid histograms and the grid outcomes the global 3-call mode keeps pending), the packed state words, the stone windows, the grid bins and -- with
 * include_stones -- the stone rows (needed whenever stones can change: regeneration extensions, or a restore into a
 * fresh handle).  as_restore puts it back; a run continued from a restored snapshot is bit-identical to the
 * uninterrupted one (same seed / env_id_offset / num_envs).  Stream-ordered, no synchronisation. */
int64_t as_snapshot_bytes(const AsHandle* h, int32_t include_stones);
int as_snapshot(AsHandle* h, void* dst, int32_t include_stones, void* stream);
int as_restore(AsHandle* h, const void* src, int32_t include_stones, void* stream);

/* Stone poses in the layout PhysX takes them (SURVEY 8 f4).  Replaces the egress of `_generate_foot_steps`,
 * ENV:119-120 -> RigidObjectCollection.write_object_pose_to_sim, rigid_object_collection.py:295-301: instead of
 * cat((steps_pos, [1,0,0,0])) -> scatter into object_state_w -> clone + convert_quat(to="xyzw") of the WHOLE (N,S,7)
 * tensor -> einsum transpose (reshape_data_to_view, :650-659), the kernel writes, for the k listed envs only, the rows
 * `view_poses[s*N + e] = (x, y, z, 0, 0, 0, 1)` of the object-major (S*N,7) x,y,z,w tensor and the index list
 * `view_ids[s*k + i] = s*N + env_ids[i]` (_env_obj_ids_to_view_ids, :675), S = AsParams.num_steps -- the two arguments of
 * root_physx_view.set_transforms(view_poses, indices=view_ids).  env_ids == NULL: all envs (k = N, in order).
 * view_ids may be NULL. */
int as_export_stone_poses(AsHandle* h, const int32_t* env_ids, int64_t n_ids, float* view_poses, int32_t* view_ids,
                          void* stream);

/* ---- grid curriculum (EXTENSION: AS_FLAG_GRID_CURRICULUM; no reference counterpart, specification in
 * oracle/grid_curriculum.py) --------------------------------------------------------------------------------------
 * With the flag set, every env that resets -- in as_step_fused, or in as_reset on the 3-call path -- has its episode
 * outcome added to a (grid_bins x grid_bins) pitch x yaw difficulty histogram, is assigned a new bin by inverse-CDF
 * sampling, and gets a stone sequence regenerated at that bin's difficulty, its stone window rebuilt at index 1.
 * as_grid_state copies the per-env bins (N bytes) and the two histograms (attempts[256] then successes[256], uint32)
 * out of / into the device state; NULL = skip.  Precondition on what is copied in: successes[b] <= attempts[b] for
 * every bin, and every bin < grid_bins * grid_bins (a larger one would index the difficulty tables past their end);
 * the library does not check it.  When a step's outcomes would carry a bin's attempts past 2^32 - 1, the bin is
 * halved first (attempts >> 1, successes >> 1), which keeps its success ratio.
 * Bins drawn in step t use the histograms as they stand after step t-1; the outcomes of step t are added when the step
 * is closed: by as_finish_step -- summed over all shards when the step is closed on a global record, so that sharded
 * runs sample from the same CDF as one handle holding all envs -- or, on the 3-call path, by as_step_pass2.  On the
 * 3-call path the histograms are shard-local (as its promotion rule is): each shard samples from its own outcomes --
 * unless the handle is in the global 3-call mode (as_peer_three_call).  There as_step_pass2 leaves the step's outcomes
 * pending, and the exchange of the NEXT as_step_pass1 (or reset outside a step) adds them, summed over all shards,
 * before anything draws from the histograms.  So between steps the histograms as_grid_state copies out lag one step
 * behind those of one handle holding all envs; right after each as_step_pass1 they are equal.
 * The draws of as_reset are made at the step counter as_step_pass1 advanced to, so bins and stones differ from those
 * of a fused step on the same inputs.  A step in which nothing resets (as_step_no_reset, or an empty device-side list)
 * records nothing.  A reset outside a step (as_reset with no as_step_pass1 before it: DirectRLEnv.reset()) ends no
 * episode: the envs draw new bins and stones but no outcome is recorded -- at start-up that would count every env as a
 * failure of bin 0 and push the sampler away from the easiest bin before training begins. */
int as_grid_state(AsHandle* h, uint8_t* bins_dst, const uint8_t* bins_src, uint32_t* hist_dst, const uint32_t* hist_src,
                  void* stream);

/* Measurement hook: two `cudaEvent_t` (as void*) that as_step_fused records on its stream immediately before and
 * after the launch of the fused step kernel alone (bench.py times the dominant kernel with them); NULL = off. */
int as_set_timing_events(AsHandle* h, void* start_event, void* stop_event);

/* Development aid: per-phase clock64() sums of the step kernel (all zero unless the library was built with
 * -DAS_TIMING); copies 16 counters to the host and optionally clears them.  Synchronises `stream`. */
int as_debug_timing(AsHandle* h, uint64_t* host16, int reset, void* stream);

/* Host-side introspection used by the tests: number of kernel launches issued by this handle so far, and
 * sizeof() of the public structs (0 AsParams, 1 AsStateIn, 2 AsStepOut, 3 AsResetOut, 4 AsStats, 5 AsMdpState,
 * 6 AsMirrorJob)
 * so that a foreign-language binding can verify its struct layout. */
int64_t as_launch_count(const AsHandle* h);
int64_t as_sizeof(int32_t which);

#ifdef __cplusplus
}
#endif
#endif /* ALLSTEPS_B200_H_ */
