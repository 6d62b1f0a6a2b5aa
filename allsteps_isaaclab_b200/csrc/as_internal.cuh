// Internal layout shared by the Allsteps kernels and the C-ABI glue (not part of the public header).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/allsteps_b200.h"

namespace as {

constexpr int kJ = AS_NUM_JOINTS;
constexpr int kS = AS_NUM_STONES;  // the default course length; a handle's own is AsParams::num_steps (normalised by as_create)
constexpr int kObs = AS_OBS_DIM;
#ifndef AS_KTILE
#define AS_KTILE AS_TILE_ENVS
#endif
constexpr int kTile = AS_KTILE;  // envs per CTA (two threads per env)
constexpr int kMaxGridBins = 256;    // grid curriculum: up to 16 x 16 bins
constexpr int kSlots = 32;           // replicated statistic accumulators (spreads same-address atomics)

// Per-step counters accumulated by the step kernels (index into Ctrl::slots[slot][]).
enum Counter {
  kCntReset = 0,
  kCntTerminated,
  kCntTimeOut,
  kCntFell,
  kCntSoFast,
  kCntDied,
  kCntAdvanced1,  // index advances in pass 1
  kCntAdvanced2,  // index advances in pass 2 (void when the fix-up discards pass 2)
  kCntSumIndex,   // sum of curr_target_index after pass 1 (numerator of ENV:471)
  kCntRegen,
  kCntLevelMax,   // max curriculum level seen (combined with max, not add)
  kCntMissed,     // AS_FLAG_MISSED_STEP: envs terminated by a missed step
  kNumCounters = 12
};

// Per-joint constants of MATH:22-40 scale_transform, precomputed by as_create.
// One 16-byte record per joint, so that the three constants of a joint reach the uniform registers with ONE constant
// load (LDCU.128) instead of three.
struct alignas(16) JointConsts {
  float4 c[AS_NUM_JOINTS];  // .x offset = (lower + upper) * 0.5   .y (upper - lower) / 2   .z 2 * RN(1 / (upper - lower))
                            // .w 0.99, the at-limit threshold of ENV:367 (so that all four words are used and load as one)
  int32_t exact_div;        // 1: use true divisions (a joint range, or step_dt, has an all-ones significand)
};

// Packed per-env MDP state word (state.x); state.y holds the bits of `potentials`.
//   [0:5) curr_target_index   [5] swing_leg   [6:8) target_reach_count   [8:12) curriculum level
//   [12:32) episode_length
// prev/next target index are always clamp(curr -/+ 1) in the reference (ENV:76-77,446-456,493-494), so they are
// derived, not stored.  old_potentials is dead between passes (overwritten at ENV:415 before it is read).
__host__ __device__ inline uint32_t pack_state(int idx, int leg, int count, int level, int ep) {
  return static_cast<uint32_t>(idx) | (static_cast<uint32_t>(leg) << 5) | (static_cast<uint32_t>(count) << 6) |
         (static_cast<uint32_t>(level) << 8) | (static_cast<uint32_t>(ep) << 12);
}
__host__ __device__ inline int state_idx(uint32_t w) { return static_cast<int>(w & 31u); }
__host__ __device__ inline int state_leg(uint32_t w) { return static_cast<int>((w >> 5) & 1u); }
__host__ __device__ inline int state_count(uint32_t w) { return static_cast<int>((w >> 6) & 3u); }
__host__ __device__ inline int state_level(uint32_t w) { return static_cast<int>((w >> 8) & 15u); }
__host__ __device__ inline int state_ep(uint32_t w) { return static_cast<int>(w >> 12); }
constexpr int kMaxEpisodeLength = (1 << 20) - 2;

// The stone window: a validated cache of the four stones around `curr_target_index` so that the step reads one
// coalesced 64-byte record per env instead of three scattered 16-byte gathers out of the S x 16-byte stone row.
// It is valid iff the tag equals the env's current index; every writer of the index or of the stones rewrites it,
// and a reader that finds a stale tag falls back to gathering from `stones` (which is always authoritative).
// S: the handle's course length.
__device__ __forceinline__ int window_slot_stone(int idx, int slot, int S) { return min(max(idx - 1 + slot, 0), S - 1); }

// Device control block at the head of the workspace.
struct Ctrl {
  uint32_t parity;        // state buffer holding the CURRENT MDP state (fused path ping-pongs)
  uint32_t promote_cur;   // level promotion decided last step, applied when the state word is next read
  uint32_t blocks_done;   // ticket counter for "last block folds the statistics"
  uint32_t blocks_done2;  // same, for the fix-up / finish kernel
  uint32_t n_reset_list;  // entries of reset_ids written this step
  uint32_t n_regen_list;  // entries of regen_ids written this step
  uint32_t fixup_ran;     // diagnostics: how many steps needed the no-reset fix-up
  uint32_t last_adv2;     // pass-2 index advances of the last step (discarded again if the fix-up runs)
  uint32_t stats_folded;  // as_fold_stats already folded this step's counters (the finish kernel must not redo it)
  uint32_t peer_epoch;    // steps closed through the peer exchange (its flag value is peer_epoch + 1, never 0)
  unsigned long long step_counter;
  AsStats stats;          // folded statistics of the last step (this shard) ...
  unsigned int grid_delta_att[kMaxGridBins];   // ... followed by this step's grid outcomes: together one AsExchange
  unsigned int grid_delta_succ[kMaxGridBins];
  unsigned int slots[kSlots][kNumCounters];
  float slot_reward[kSlots];
  unsigned int grid_attempts[kMaxGridBins];   // grid curriculum extension: episodes ended per difficulty bin
  unsigned int grid_successes[kMaxGridBins];  // ... of which the env had passed half of the stones
  unsigned long long dbg_t[16];               // -DAS_TIMING builds only: summed clock64() phase durations per CTA
  AsExchange gx;                              // exchange records summed over all shards (peer exchange)
  unsigned long long peer_timeouts;           // peers that did not deliver within the time limit (sticky: see peer_error)
  uint32_t peer_error;                        // != 0: a peer exchange timed out; the shards may have diverged (AS_ERR_PEER)
  uint32_t step_state;                        // written by the LAST CTA of every fused step kernel: 2 = it closed the step itself
                                              // (statistics folded, promotion decided, parity flipped), 1 = k_fixup_finish has to
  uint32_t any_reset;                         // global 3-call mode: pass 1 flagged an env on some shard this step (written by
                                              // k_peer_exchange; read by k_pass2_commit / k_pass2_revert, DRL:359-360)
};
// (the control block's slot in the workspace and the snapshot stays 8448 bytes: checkpoints keep their layout)
static_assert(sizeof(Ctrl) <= 8448, "Ctrl must fit its 8448-byte workspace slot");

static_assert(offsetof(Ctrl, grid_delta_att) == offsetof(Ctrl, stats) + sizeof(AsStats) &&
                  offsetof(Ctrl, grid_delta_succ) == offsetof(Ctrl, grid_delta_att) + sizeof(unsigned int) * kMaxGridBins,
              "Ctrl::stats and the grid outcome arrays form one AsExchange");
// (mdp.py reads the histograms in place at this distance behind the statistics: _cabi.GRID_HIST_OFFSET)
static_assert(offsetof(Ctrl, grid_attempts) == offsetof(Ctrl, stats) + sizeof(AsExchange) + 1664 &&
                  offsetof(Ctrl, grid_successes) == offsetof(Ctrl, grid_attempts) + sizeof(unsigned int) * kMaxGridBins,
              "the difficulty-grid histograms sit 1664 bytes behind the exchange record");

// One bin's step outcomes (da, ds) join its histogram counters (oracle/grid_curriculum.py, "fold"): a bin whose
// attempts would pass 2^32 - 1 is halved first, which keeps its success ratio and successes <= attempts.  A step's
// delta is below 2^31 (at most the run's env count), so one halving makes room.  Single writer: the closing CTA.
__device__ __forceinline__ void grid_fold(unsigned int& att, unsigned int& succ, unsigned int da, unsigned int ds) {
  if (static_cast<unsigned long long>(att) + da > 0xFFFFFFFFull) {
    att >>= 1;
    succ >>= 1;
  }
  att += da;
  succ += ds;
}

// Peer exchange buffer of one rank: for each of the two epoch parities one 128-byte slot per sending rank.
constexpr int kMaxPeers = AS_MAX_PEERS;
constexpr int kPeerCounters = 10;  // the additive head of AsStats
struct PeerSlot {
  unsigned long long flag;  // epoch the counters belong to; written last (release), polled by the owner
  long long counters[kPeerCounters];
  unsigned long long pad[5];
};
static_assert(sizeof(PeerSlot) == 128, "one slot per 128-byte line");
struct PeerGrid {  // one sender's grid outcomes of a step
  unsigned int att[kMaxGridBins], succ[kMaxGridBins];
};
constexpr int64_t kPeerGridOffset = 2 * kMaxPeers * static_cast<int64_t>(sizeof(PeerSlot));
constexpr int64_t kPeerBufferBytes = kPeerGridOffset + 2 * kMaxPeers * static_cast<int64_t>(sizeof(PeerGrid));
static_assert(offsetof(AsExchange, grid_attempts) == sizeof(AsStats), "AsExchange is AsStats + the two grid arrays");
struct PeerArgs {
  PeerSlot* buf[kMaxPeers];  // buf[r]: rank r's buffer as seen from this GPU (own: local pointer, others: IPC mappings)
  int32_t world, rank;
  unsigned long long timeout_ns;  // how long to poll for a peer's counters; 0 = without limit
  uint32_t* host_error;           // mapped pinned host word, set to the epoch when a peer timed out (read by the API, no sync)
};

struct Workspace {
  Ctrl* ctrl;
  uint2* state[2];    // (N) packed state / potentials, ping-pong
  float4* stones;     // (N,S) x,y,z (world frame), cumulative yaw; S = AsParams::num_steps
  float4* window;     // (N,4) cache of stones idx-1, idx, idx+1, idx+2 (clamped); entry 0's .w holds idx as a tag
  int32_t* reset_ids; // (N)
  int32_t* regen_ids; // (N)
  uint8_t* regen_info;// (N) curr_target_index at the end of the episode, parallel to regen_ids (grid curriculum)
  uint8_t* bin;       // (N) difficulty-grid bin of each env (grid curriculum extension)
  uint8_t* contact_pre;// (N) ENV:425 evaluated by k_prepare*: bit 0 / 1 = the right / left foot presses on the env's CURRENT stone
                      // (|F| > contact_epsilon), bit 2 / 3 = on the stone after it (what pass 2 needs when pass 1 advances)
  float* body_dense;  // (N,3,3) right foot, left foot, torso positions gathered out of a strided body tensor (k_prepare*)
  float4* tail1;      // (N,3) 3-call path: the observation tail (foot contacts, targets_b: columns 48..58) as pass 1 leaves it
  uint8_t* pass1_reset;// (N) 3-call path: the env was flagged for reset by pass 1 (terminated | time_out)
  uint32_t* win_stale;// (ceil(N/32)) one bit per env: its stone-window record must be refreshed by k_prepare* (set by the
                      // step kernel instantiation that does not write windows; set for every env of a fresh handle)
};

struct WorkspaceLayout {
  int64_t ctrl_off, state0_off, state1_off, stones_off, window_off, reset_ids_off, regen_ids_off, regen_info_off,
      bin_off, contact_pre_off, body_dense_off, tail1_off, pass1_reset_off, win_stale_off, total;
};

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// S: the handle's course length (the stone rows are the only part that depends on it)
inline WorkspaceLayout workspace_layout(int64_t n, int S) {
  WorkspaceLayout l;
  int64_t off = 0;
  l.ctrl_off = off;
  off = align_up(off + static_cast<int64_t>(sizeof(Ctrl)), 256);
  l.state0_off = off;
  off = align_up(off + n * 8, 256);
  l.state1_off = off;
  off = align_up(off + n * 8, 256);
  l.stones_off = off;
  off = align_up(off + n * S * 16, 256);
  l.window_off = off;
  off = align_up(off + n * 4 * 16, 256);
  l.reset_ids_off = off;
  off = align_up(off + n * 4, 256);
  l.regen_ids_off = off;
  off = align_up(off + n * 4, 256);
  l.regen_info_off = off;
  off = align_up(off + n, 256);
  l.bin_off = off;
  off = align_up(off + n, 256);
  l.contact_pre_off = off;
  off = align_up(off + n, 256);
  l.body_dense_off = off;
  off = align_up(off + n * 36, 256);
  l.tail1_off = off;
  off = align_up(off + n * 48, 256);
  l.pass1_reset_off = off;
  off = align_up(off + n, 256);
  l.win_stale_off = off;
  off = align_up(off + (n + 31) / 32 * 4, 256);
  l.total = off;
  return l;
}

enum StepMode { kModeFused = 0, kModeFixup = 1, kModePass1 = 2, kModePass2 = 3 };

struct StepArgs {
  AsParams P;
  JointConsts jc;
  AsStateIn in;
  const float* actions;
  int64_t actions_stride;
  AsStepOut out;
  // AsStepOut.final_obs moved the fields behind `out` by 8 bytes; ptxas then allocated the FAST pass-1 instantiations
  // differently (more spills).  Moving them by 16 keeps their 16-byte alignment as it was, and that code as it was.
  uint64_t pad_final_obs;
  Workspace ws;
  const int64_t* ext_episode_length;  // 3-call path: DirectRLEnv-owned counter (already incremented), or null
  const AsExchange* global_stats;     // fix-up/finish: exchange record summed over ranks, or null
  int64_t num_envs;
  int64_t env_id_offset;
  int32_t num_tiles;
  int32_t tile_base;                  // first tile of this launch (k_step: 0 for the full tiles, the last tile's index for a ragged tail)
  int32_t want_reset_list;            // fused: compact the ids of the envs that reset
  int32_t use_pre;                    // 1: contact norms come from k_prepare* (large batches), 0: gather here
  int32_t self_finish;                // fused: the last CTA closes the step when at least one env reset (no peers, no regeneration)
  int32_t pdl_wait;                   // 1: launched as a programmatic dependent of k_prepare*
  int32_t body_from_prepare;          // 1: in.body_pos is the dense array k_prepare* of this step writes
  uint32_t dense16;                   // per-array "dense and 16-byte aligned" bits (DenseBit), evaluated by the host
  float inv_step_dt;                  // RN(1 / P.step_dt) for the two-FMA quotient of ENV:416 (see JointConsts::exact_div)
  AsResetOut rows;                    // fused: start-pose rows for PhysX, written at the env's own row (optional)
  PeerArgs peer;                      // fused + self_finish with peers connected: the last CTA exchanges the counters itself
};

struct ResetArgs {
  AsParams P;
  Workspace ws;
  AsResetOut out;
  const float* env_origins;
  const int32_t* env_ids;   // 3-call path: explicit list; fused path: null (uses ws.reset_ids / ws.regen_ids)
  int64_t n_ids;
  int64_t* ext_episode_length;
  const AsExchange* global_stats;
  const float* stone_uniforms;  // optional explicit draws (5,N,S)
  int64_t num_envs;
  int64_t env_id_offset;
  int32_t fused;                // 1: state words were already reset by the step kernel, rows go to env's own row
  int32_t into_other;           // 3-call path behind a speculating pass 1: the reset state words go into the OTHER buffer
  int32_t force_any_reset;      // 3-call path: an explicit id list means `_reset_idx` was entered, i.e. some env reset
  int32_t peer_decided;         // global 3-call mode: k_peer_exchange already decided the promotion on the global sums
};

}  // namespace as
