// Kernels (b) and (c) plus the small adapters around the fused step:
//   k_reset_list      3-call path: start-pose rows for PhysX (ENV:505-565) from the same Philox draws the step kernel
//                     uses, MDP words, the list of envs to regenerate, for an explicit / device-compacted id list
//   k_reset_rows      grid-curriculum turnover + stone-sequence regeneration (ENV:106-174) for the envs the fused step
//                     kernel or k_reset_list listed
//   k_generate_stones stone sequences for all / listed envs (init, ENV:71)
//   k_apply_action    ENV:257-274
//   k_mirror_batch    ENV:570-660 (mirror-symmetry augmentation; 128-row tiles through shared memory by TMA bulk copies)
//   k_export / k_import  packed state <-> the reference's int64/fp32 buffers
#pragma once
#include "as_internal.cuh"
#include "as_math.cuh"
#include "philox.cuh"
#include "as_step_kernel.cuh"

namespace as {

constexpr unsigned kFullMask = 0xffffffffu;

// Sequential inclusive scan over the first S lanes, accumulated in double exactly like torch.cumsum on CPU
// (acc_type<float> is double there) -- a log-step warp scan would re-associate the additions.
__device__ __forceinline__ float warp_cumsum_sequential(float x, int lane, int S) {
  double acc = 0.0;
  float mine = 0.0f;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const float vs = __shfl_sync(kFullMask, x, s);
    acc += static_cast<double>(vs);
    if (lane == s) mine = static_cast<float>(acc);
  }
  return mine;
}

// How hard an env's stone sequence is: the reference has one scalar ratio = level / max_level for yaw and pitch and
// a per-level upper bound of the stone distance (ENV:126-133); the grid-curriculum extension has one ratio per axis.
struct Difficulty {
  float ratio_yaw, ratio_pitch, dist_upper;
};
__device__ __forceinline__ Difficulty difficulty_of_level(const AsParams& P, int level) {
  level = min(level, P.max_level);                                                   // ENV:126
  const float ratio = static_cast<float>(level) / static_cast<float>(P.max_level);   // ENV:127
  return Difficulty{ratio, ratio, P.dist_upper[level]};
}
// bin = i * B + j (i: pitch bin, j: yaw bin); see oracle/grid_curriculum.py for the definition
__device__ __forceinline__ Difficulty difficulty_of_bin(const AsParams& P, int bin) {
  const int B = static_cast<int>(P.grid_bins);
  const int i = bin / B, j = bin - i * B;
  const float denom = static_cast<float>(B - 1);
  const int k = (max(i, j) * P.max_level) / (B - 1);
  return Difficulty{static_cast<float>(j) / denom, static_cast<float>(i) / denom, P.dist_upper[k]};
}
__device__ __forceinline__ Difficulty difficulty_of_env(const AsParams& P, const Workspace& ws, int64_t e, int level) {
  return (P.flags & AS_FLAG_GRID_CURRICULUM) ? difficulty_of_bin(P, ws.bin[e]) : difficulty_of_level(P, level);
}

// ENV:125-174 for one env, one stone per lane (lanes >= S idle).  `u_dr/u_dphi/u_dtheta` are this lane's draws.
// S: the course length (a compile-time constant where the caller knows it is the default).
__device__ __forceinline__ void generate_stones_warp(const AsParams& P, int lane, const Difficulty& D,
                                                     const Vec3& origin, float u_dr, float u_dphi, float u_dtheta,
                                                     float4* out_row, int S) {
  const float deg2rad = 0.017453292519943295f;  // torch.deg2rad multiplies by float32(pi/180)
  const float half_pi = 1.5707963705062866f;
  const float yaw_lo = (P.yaw_range_deg[0] * D.ratio_yaw) * deg2rad, yaw_hi = (P.yaw_range_deg[1] * D.ratio_yaw) * deg2rad;
  const float pit_lo = (P.pitch_range_deg[0] * D.ratio_pitch) * deg2rad + half_pi;   // ENV:132
  const float pit_hi = (P.pitch_range_deg[1] * D.ratio_pitch) * deg2rad + half_pi;
  float dr = torch_lerp(P.dist_lower, D.dist_upper, u_dr);                           // ENV:137
  float dphi = torch_lerp(yaw_lo, yaw_hi, u_dphi);                                   // ENV:138
  float dth = torch_lerp(pit_lo, pit_hi, u_dtheta);                                  // ENV:139
  if (lane == 0) {                                                                   // ENV:144-146
    dr = 0.0f; dphi = 0.0f; dth = half_pi;
  } else if (lane <= 2) {                                                            // ENV:148-150
    dr = P.init_step_separation; dphi = 0.0f; dth = half_pi;
  }
  if (lane >= S) { dr = 0.0f; dphi = 0.0f; dth = half_pi; }
  const float phi = warp_cumsum_sequential(dphi, lane, S);                              // ENV:155
  const float st = sinf(dth), ct = cosf(dth);
  const float dx = (dr * st) * cosf(phi);                                            // ENV:157
  const float dy = (dr * st) * sinf(phi);                                            // ENV:158
  const float dz = dr * ct;                                                          // ENV:159
  const float x = warp_cumsum_sequential(dx, lane, S);                               // ENV:165-167
  const float y = warp_cumsum_sequential(dy, lane, S);
  const float z = warp_cumsum_sequential(dz, lane, S);
  if (lane < S) out_row[lane] = make_float4(x + origin.x, y + origin.y, z + origin.z, phi);  // ENV:111
}

// The same for one env by ONE thread: the S stones in sequence, the four cumulative sums as running double
// accumulators (the additions happen in the same order, so the results are those of the warp version bit for bit).
// `draw(k, s)`: uniform k (0 dr, 1 dphi, 2 dtheta) of stone s.  Used where many envs regenerate at once (the
// reset-heavy configuration): a thread per env keeps thousands of independent chains in flight where a warp per env
// spends its time in 4 x S dependent shuffle steps with 32 - S idle lanes.
template <typename Draw>
__device__ __forceinline__ void generate_stones_thread(const AsParams& P, const Difficulty& D, const Vec3& origin,
                                                       Draw draw, float4* out_row, float4* window_row, int S) {
  const float deg2rad = 0.017453292519943295f;
  const float half_pi = 1.5707963705062866f;
  const float yaw_lo = (P.yaw_range_deg[0] * D.ratio_yaw) * deg2rad, yaw_hi = (P.yaw_range_deg[1] * D.ratio_yaw) * deg2rad;
  const float pit_lo = (P.pitch_range_deg[0] * D.ratio_pitch) * deg2rad + half_pi;
  const float pit_hi = (P.pitch_range_deg[1] * D.ratio_pitch) * deg2rad + half_pi;
  double phi_acc = 0.0, x = 0.0, y = 0.0, z = 0.0;
  float4 v;
#pragma unroll 1
  for (int s = 0; s < S; ++s) {
    float dr = torch_lerp(P.dist_lower, D.dist_upper, draw(0, s));   // ENV:137
    float dphi = torch_lerp(yaw_lo, yaw_hi, draw(1, s));             // ENV:138
    float dth = torch_lerp(pit_lo, pit_hi, draw(2, s));              // ENV:139
    if (s == 0) {                                                    // ENV:144-146
      dr = 0.0f; dphi = 0.0f; dth = half_pi;
    } else if (s <= 2) {                                             // ENV:148-150
      dr = P.init_step_separation; dphi = 0.0f; dth = half_pi;
    }
    phi_acc += static_cast<double>(dphi);                            // ENV:155
    const float phi = static_cast<float>(phi_acc);
    const float st = sinf(dth), ct = cosf(dth);
    x += static_cast<double>((dr * st) * cosf(phi));                 // ENV:157,165
    y += static_cast<double>((dr * st) * sinf(phi));                 // ENV:158,166
    z += static_cast<double>(dr * ct);                               // ENV:159,167
    v = make_float4(static_cast<float>(x) + origin.x, static_cast<float>(y) + origin.y,
                           static_cast<float>(z) + origin.z, phi);   // ENV:111
    out_row[s] = v;
    if (s < 4) {  // the env restarts at index 1: window = stones 0..3, tagged
      if (s == 0) v.w = __int_as_float(1);
      window_row[s] = v;
    }
  }
  if (S < 4) window_row[3] = v;  // (slot 3 holds stone min(3, S - 1): the last one)
}

// Rebuilds one env's stone window from its stone row (lanes 0..3); call after the row was (re)written.
__device__ __forceinline__ void rebuild_window_warp(const float4* stone_row, float4* window_row, int idx, int lane,
                                                    int S) {
  __syncwarp();
  if (lane < 4) {
    float4 v = stone_row[window_slot_stone(idx, lane, S)];
    if (lane == 0) v.w = __int_as_float(idx);
    window_row[lane] = v;
  }
}

__device__ __forceinline__ void stone_draws(const ResetArgs& a, unsigned long long step, int64_t e, uint32_t gid,
                                            int lane, float& u_dr, float& u_dphi, float& u_dth, int S) {
  u_dr = u_dphi = u_dth = 0.0f;
  if (lane >= S) return;
  if (a.stone_uniforms) {  // explicit (5,N,S) tables indexed by local env id
    const int64_t plane = a.num_envs * S;
    u_dr = a.stone_uniforms[0 * plane + e * S + lane];
    u_dphi = a.stone_uniforms[1 * plane + e * S + lane];
    u_dth = a.stone_uniforms[2 * plane + e * S + lane];
  } else {
    u_dr = philox_uniform(a.P.seed, step, kStreamStones, gid, 0 * S + lane);
    u_dphi = philox_uniform(a.P.seed, step, kStreamStones, gid, 1 * S + lane);
    u_dth = philox_uniform(a.P.seed, step, kStreamStones, gid, 2 * S + lane);
  }
}

// Kernel (b) of the 3-call path (as_reset; behind the fused step the step kernel resets its envs itself).  For the
// explicit `env_ids`: resets the MDP word and the DirectRLEnv episode counter, writes the compact PhysX rows, decides
// regeneration and lists the envs that regenerate for k_reset_rows.
__global__ void __launch_bounds__(256, 3) k_reset_list(const __grid_constant__ ResetArgs a) {
  const AsParams& P = a.P;
  const int S = static_cast<int>(P.num_steps);
  Ctrl* ctrl = a.ws.ctrl;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const unsigned long long step = ctrl->step_counter;
  // n_ids < 0: the list pass 1 compacted on the device
  const int64_t n_reset = a.n_ids < 0 ? static_cast<int64_t>(ctrl->n_reset_list) : a.n_ids;
  if (!a.peer_decided && blockIdx.x == 0 && threadIdx.x == 0) {
    // 3-call path: `_reset_idx` opens with the promotion rule (ENV:471-479) on the statistics pass 1 folded.  The
    // decision is in force from here on: k_reset_rows regenerates at the promoted level (ENV:471 precedes ENV:500),
    // the next pass 1 applies it to the state words.  (Global 3-call mode: k_peer_exchange decided it on the sums.)
    AsStats s = ctrl->stats;
    if (a.force_any_reset) s.n_reset = s.n_reset > 0 ? s.n_reset : 1;
    ctrl->promote_cur = promotion_decision(P, s);
  }
  const uint32_t parity = ctrl->parity;
  // after a speculating pass 1 the step continues in the other state buffer
  uint2* st_cur = a.into_other ? a.ws.state[parity ^ 1u] : a.ws.state[parity];
  // Explicit id list (3-call path).  FOUR envs per warp, eight lanes each: a reset env is a chain of dependent loads
  // (id -> state word -> origins -> stones) with a little arithmetic in between, so a warp per env leaves the kernel
  // latency-bound at a few thousand resident warps; four independent chains per warp quadruple the loads in flight.
  const int grp = lane >> 3, g = lane & 7;
  for (int64_t w0 = warp * 4; w0 < n_reset; w0 += n_warps * 4) {
    const int64_t w = w0 + grp;
    const bool have = w < n_reset;
    int64_t e = 0;
    uint32_t word = 0;
    bool regen = false;
    if (have) {
      e = a.env_ids[w];
      const int64_t row = w;
      const uint32_t gid = static_cast<uint32_t>(e + a.env_id_offset);
      word = st_cur[e].x;
      const float ox = a.env_origins[e * 3];
      const float oy = a.env_origins[e * 3 + 1];
      const float oz = a.env_origins[e * 3 + 2];
      const uint4 b0 = philox_block(P.seed, step, kStreamReset, gid, 0);
      const bool mirror = u32_to_unit(b0.x) > 0.5f;  // ENV:518
      for (int j = g; j < kJ; j += 8) {
        float lo, hi, pose, pose_m, vel_m;
        load_reset_tables(P, j, lo, hi, pose, pose_m, vel_m);
        const float u = philox_uniform(P.seed, step, kStreamReset, gid, 1 + j);
        if (a.out.joint_pos) a.out.joint_pos[row * kJ + j] = reset_joint_value(P, mirror ? pose_m : pose, lo, hi, u);
        if (a.out.joint_vel) a.out.joint_vel[row * kJ + j] = mirror ? vel_m : 0.0f;
      }
      if (a.out.root_state) {
        const float z = mirror ? -0.0f : 0.0f;
        for (int c = g; c < AS_ROOT_STATE_DIM; c += 8) {
          float val = 0.0f;
          if (c == 0) val = P.default_root_pos[0] + ox;
          else if (c == 1) val = P.default_root_pos[1] + oy;
          else if (c == 2) val = P.default_root_pos[2] + oz;
          else if (c == 3) val = 1.0f;
          else if (c <= 6) val = z;
          a.out.root_state[row * AS_ROOT_STATE_DIM + c] = val;
        }
      }
      // the rule of the fused step kernel: every env with the grid curriculum, else those past half of their stones
      regen = (P.flags & AS_FLAG_GRID_CURRICULUM) || ((P.flags & AS_FLAG_INTENDED_REGEN) && state_idx(word) > S / 2);
      if (g == 0) {
        if (a.out.reset_ids) a.out.reset_ids[w] = static_cast<int32_t>(e);
        a.ws.reset_ids[w] = static_cast<int32_t>(e);  // (k_pass2_commit walks this list)
        uint2 sw;
        sw.x = pack_state(1, mirror ? 1 : 0, 0, state_level(word), 0);  // ENV:487-494,538; DRL:584
        sw.y = __float_as_uint(0.0f);
        st_cur[e] = sw;
        if (a.ext_episode_length) a.ext_episode_length[e] = 0;
      }
    }
    // the envs that regenerate join the list k_reset_rows (launched behind this kernel) works through: the grid
    // turnover and the stones, the same kernel as behind the fused step.  regen_info: the index the episode ended at
    // (the word as pass 1 left it -- read above, before the reset overwrote it)
    const bool listed = have && regen && g == 0;
    const unsigned lmask = __ballot_sync(kFullMask, listed);
    if (lmask) {
      const int leader = __ffs(lmask) - 1;
      unsigned base = 0;
      if (lane == leader) {
        base = atomicAdd(&ctrl->n_regen_list, static_cast<unsigned>(__popc(lmask)));
        atomicAdd(reinterpret_cast<unsigned long long*>(&ctrl->stats.n_regenerated),
                  static_cast<unsigned long long>(__popc(lmask)));
      }
      base = __shfl_sync(kFullMask, base, leader);
      if (listed) {
        const unsigned pos = base + __popc(lmask & ((1u << lane) - 1u));
        a.ws.regen_ids[pos] = static_cast<int32_t>(e);
        a.ws.regen_info[pos] = static_cast<uint8_t>(state_idx(word));
      }
    }
    if (have && !regen && g < 4) {  // the env restarts at index 1 on its stones: its stone window
      float4 v = a.ws.stones[e * S + window_slot_stone(1, g, S)];
      if (g == 0) v.w = __int_as_float(1);
      a.ws.window[e * 4 + g] = v;
    }
  }
  if (a.out.n_reset && blockIdx.x == 0 && threadIdx.x == 0) *a.out.n_reset = static_cast<int32_t>(n_reset);
  // (the count of the list k_pass2_commit walks.  Outside a step no commit follows to clear it, and the next fused step
  // would start its reset-id list behind it, past the end of the N-entry buffers)
  if (a.into_other && blockIdx.x == 0 && threadIdx.x == 0) ctrl->n_reset_list = static_cast<uint32_t>(n_reset);
}


// ------------------------------------------------------------------------------------------------ kernels (b) + (c)
// Everything that happens to the envs listed for regeneration, in ONE launch: behind the fused step the step kernel
// listed them (fused = 1), on the 3-call path k_reset_list did (fused = 0; there the draws are at the step counter
// pass 1 or k_prepare_reset advanced to, the outcomes join the histograms when k_pass2_commit closes the step -- in
// the global 3-call mode when the next k_peer_exchange has summed them over the shards -- and a reset outside a step
// -- into_other = 0 -- records none).
//   (c) grid-curriculum extension (no reference counterpart; specification = oracle/grid_curriculum.py): the outcome of
//       the episode that just ended is recorded against the bin the env WAS playing -- a shared-memory histogram per
//       CTA, flushed with one atomic per touched bin into the step's outcome record (Ctrl::grid_delta_*), which joins
//       the histograms when the step is closed, summed over the shards first when the run is sharded -- and the env
//       draws its new bin by inverse-CDF search in the integer CDF of the bin weights (histograms as they stand after
//       the PREVIOUS step; every CTA rebuilds the CDF with a shuffle scan).
//   (b) the stone row (ENV:106-174) and the stone window of the env, at the new difficulty.
// Two shapes of the same arithmetic (bit-identical: same draws, same order of the additions), chosen by the host from
// the batch size: one WARP per env for small batches, where the list is a few hundred envs and the kernel is pure
// latency -- the S stones' draws, interpolations and sines run side by side -- and one THREAD per env for large
// ones, where thousands of independent chains in flight beat 4 x S dependent shuffle steps with 32 - S idle lanes
// (BASELINE config 5: 257 000 of 1 M envs regenerate per step).
constexpr uint32_t kStreamGrid = 2;

// 1 + 1024 s (a - s) / (a^2 + 1), exact for every s <= a < 2^32: s (a - s) < 2^62 and a^2 + 1 < 2^64 fit 64 bits,
// the product with 1024 does not.  The quotient has ten bits (every weight is in 1..256), so it is formed by ten
// steps of binary long division; s (a - s) < a^2 + 1 keeps every partial remainder below the divisor.
__device__ __forceinline__ unsigned int grid_weight(unsigned int a, unsigned int s) {
  if (a == 0) return 256u;  // unvisited bins are tried
  const unsigned long long A = a, S = s, den = A * A + 1ull;
  unsigned long long rem = S * (A - S);
  unsigned int q = 0;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const bool carry = (rem >> 63) != 0;  // 2 rem passes 2^64: it exceeds den, and the wrapped difference is exact
    rem <<= 1;
    q <<= 1;
    if (carry || rem >= den) {
      rem -= den;
      q |= 1u;
    }
  }
  return 1u + q;  // peaks at a 50 % success rate
}

// DEFAULT_S: the handle runs courses of the default length, which the generators then take as a constant.
template <bool BY_WARP, bool DEFAULT_S>
__global__ void __launch_bounds__(256, 4) k_reset_rows(const __grid_constant__ ResetArgs a) {
  __shared__ unsigned int s_cdf[kMaxGridBins], s_att[kMaxGridBins], s_succ[kMaxGridBins];
  __shared__ unsigned int s_warp_tot[8];
  asm volatile("griddepcontrol.launch_dependents;");  // the finish kernel may become resident; it waits for us
  asm volatile("griddepcontrol.wait;" ::: "memory");  // the step kernel has completed: its id lists are final
  const AsParams& P = a.P;
  const int S = DEFAULT_S ? kS : static_cast<int>(P.num_steps);
  Ctrl* ctrl = a.ws.ctrl;
  const int t = threadIdx.x, lane = t & 31, warp_in_cta = t >> 5;
  const int64_t n_regen = ctrl->n_regen_list;
  const int64_t n_threads = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t n_warps = n_threads >> 5;
  // (block-uniform: CTAs without a list entry leave before the first barrier)
  if (static_cast<int64_t>(blockIdx.x) * (BY_WARP ? blockDim.x >> 5 : blockDim.x) >= n_regen) return;
  const bool grid = (P.flags & AS_FLAG_GRID_CURRICULUM) != 0;
  const int nb = static_cast<int>(P.grid_bins * P.grid_bins);
  if (grid) {
    // inclusive prefix sum of the bin weights: shuffle scan inside each warp, then the warp totals
    unsigned int v = t < nb ? grid_weight(__ldcg(&ctrl->grid_attempts[t]), __ldcg(&ctrl->grid_successes[t])) : 0u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int up = __shfl_up_sync(kFullMask, v, o);
      if (lane >= o) v += up;
    }
    if (lane == 31) s_warp_tot[warp_in_cta] = v;
    s_att[t] = 0u;
    s_succ[t] = 0u;
    __syncthreads();
    unsigned int base = 0;
    for (int w = 0; w < warp_in_cta; ++w) base += s_warp_tot[w];
    s_cdf[t] = v + base;
    __syncthreads();
  }
  const unsigned long long step = ctrl->step_counter;
  // a reset outside a step (3-call path without a pass 1: DirectRLEnv.reset()) ends no episode: new bins, no outcomes
  const bool record = a.fused || a.into_other;
  // outcome of list entry w (env e) against the bin it played, then the new bin of the env
  auto grid_turnover = [&](int64_t w, int64_t e) -> int {
    const int b0 = a.ws.bin[e];
    if (record && BY_WARP) {  // a short list spread over many CTAs: straight into the step's outcome record
      atomicAdd(&ctrl->grid_delta_att[b0], 1u);
      if (a.ws.regen_info[w] > S / 2) atomicAdd(&ctrl->grid_delta_succ[b0], 1u);
    } else if (record) {
      atomicAdd(&s_att[b0], 1u);
      if (a.ws.regen_info[w] > S / 2) atomicAdd(&s_succ[b0], 1u);
    }
    const unsigned long long total = s_cdf[nb - 1];
    const uint4 blk = philox_block(P.seed, step, kStreamGrid, static_cast<uint32_t>(e + a.env_id_offset), 0);
    const unsigned long long target = (static_cast<unsigned long long>(blk.x >> 8) * total) >> 24;
    int lo = 0, hi = nb - 1;  // first bin with cdf > target
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (s_cdf[mid] > target) hi = mid; else lo = mid + 1;
    }
    a.ws.bin[e] = static_cast<uint8_t>(lo);
    return lo;
  };
  // promotion decided in THIS step is already in force when stones are regenerated (ENV:471 precedes ENV:500)
  int promote_now;
  if (!a.fused) {  // 3-call path: k_reset_list, launched before, decided it
    promote_now = static_cast<int>(ctrl->promote_cur);
  } else if (a.global_stats) {
    promote_now = static_cast<int>(promotion_decision(P, a.global_stats->stats));
  } else {  // the step kernel's counters are still in the replicated slots (folded by the finish kernel)
    const unsigned nr = slot_sum(ctrl, kCntReset);
    const unsigned si = slot_sum(ctrl, kCntSumIndex);
    promote_now = static_cast<int>(promotion_rule(P, nr, si, a.num_envs));
  }
  // the state words as reset: the fused step and a speculating pass 1 wrote the other buffer, a reset outside a step
  // the current one
  const uint2* st_cur = a.ws.state[record ? ctrl->parity ^ 1u : ctrl->parity];
  if (BY_WARP) {
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + t) >> 5;
    for (int64_t w = warp; w < n_regen; w += n_warps) {
      const int64_t e = a.ws.regen_ids[w];
      int bin = 0;
      if (grid) {
        if (lane == 0) bin = grid_turnover(w, e);
        bin = __shfl_sync(kFullMask, bin, 0);
      }
      const int level = min(state_level(st_cur[e].x) + promote_now, P.max_level);
      const Vec3 origin{a.env_origins[e * 3], a.env_origins[e * 3 + 1], a.env_origins[e * 3 + 2]};
      const Difficulty D = grid ? difficulty_of_bin(P, bin) : difficulty_of_level(P, level);
      float u0, u1, u2;
      stone_draws(a, step, e, static_cast<uint32_t>(e + a.env_id_offset), lane, u0, u1, u2, S);
      generate_stones_warp(P, lane, D, origin, u0, u1, u2, a.ws.stones + e * S, S);
      rebuild_window_warp(a.ws.stones + e * S, a.ws.window + e * 4, 1, lane, S);  // the env restarts at index 1
    }
  } else {
    const int64_t tid = static_cast<int64_t>(blockIdx.x) * blockDim.x + t;
    for (int64_t w = tid; w < n_regen; w += n_threads) {
      const int64_t e = a.ws.regen_ids[w];
      const uint32_t gid = static_cast<uint32_t>(e + a.env_id_offset);
      const int bin = grid ? grid_turnover(w, e) : 0;
      const int level = min(state_level(st_cur[e].x) + promote_now, P.max_level);
      const Vec3 origin{a.env_origins[e * 3], a.env_origins[e * 3 + 1], a.env_origins[e * 3 + 2]};
      const Difficulty D = grid ? difficulty_of_bin(P, bin) : difficulty_of_level(P, level);
      if (a.stone_uniforms) {
        const int64_t plane = a.num_envs * S;
        const float* tab = a.stone_uniforms + e * S;
        generate_stones_thread(P, D, origin, [&](int k, int s) { return tab[k * plane + s]; }, a.ws.stones + e * S,
                               a.ws.window + e * 4, S);
      } else {
        // draw d = k * S + s is component d & 3 of Philox block d >> 2.  blk[k] holds the block of draw k * S + s; the
        // three are fetched together whenever one of them enters a new block (S = 20: every fourth stone, blocks
        // 5 k + (s >> 2) -- three blocks serve four stones)
        uint4 blk[3];
        generate_stones_thread(P, D, origin, [&](int k, int s) {
          if (k == 0 && (s == 0 || (s & 3) == 0 || ((S + s) & 3) == 0 || ((2 * S + s) & 3) == 0)) {
#pragma unroll
            for (int q = 0; q < 3; ++q) blk[q] = philox_block(P.seed, step, kStreamStones, gid, static_cast<uint32_t>((q * S + s) >> 2));
          }
          return u32_to_unit(lane_of(blk[k], (k * S + s) & 3)); }, a.ws.stones + e * S, a.ws.window + e * 4, S);
      }
    }
  }
  if (grid && !BY_WARP) {
    __syncthreads();
    if (s_att[t]) atomicAdd(&ctrl->grid_delta_att[t], s_att[t]);
    if (s_succ[t]) atomicAdd(&ctrl->grid_delta_succ[t], s_succ[t]);
  }
}

// Stone sequences for all envs (env_ids == null) or a list; level from the packed word (+ pending promotion).
__global__ void __launch_bounds__(256) k_generate_stones(const __grid_constant__ ResetArgs a) {
  Ctrl* ctrl = a.ws.ctrl;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t n = a.env_ids ? a.n_ids : a.num_envs;
  const unsigned long long step = ctrl->step_counter;
  const uint2* st = a.ws.state[ctrl->parity];
  const int pending = static_cast<int>(ctrl->promote_cur);
  for (int64_t w = warp; w < n; w += n_warps) {
    const int64_t e = a.env_ids ? a.env_ids[w] : w;
    const uint32_t gid = static_cast<uint32_t>(e + a.env_id_offset);
    const int level = min(state_level(st[e].x) + pending, a.P.max_level);
    const Vec3 origin{a.env_origins[e * 3], a.env_origins[e * 3 + 1], a.env_origins[e * 3 + 2]};
    float u0, u1, u2;
    const int S = static_cast<int>(a.P.num_steps);
    stone_draws(a, step, e, gid, lane, u0, u1, u2, S);
    generate_stones_warp(a.P, lane, difficulty_of_env(a.P, a.ws, e, level), origin, u0, u1, u2, a.ws.stones + e * S, S);
    rebuild_window_warp(a.ws.stones + e * S, a.ws.window + e * 4, state_idx(st[e].x), lane, S);
  }
}

// ENV:257-274: efforts = gain[level] * gear * clamp(action).  Runs four times per env step (decimation, CFG:55), a pure
// stream of 84 bytes in and 84 bytes out per env: full 128-env tiles are brought in by one TMA bulk copy, scaled in
// place in shared memory (the env's gain from its state word, the gears from a shared copy of the table -- out of the
// constant bank a warp's 21 different joints would be 21 serialised reads) and sent out by one bulk copy; the envs
// behind the last full tile, and action views that are strided or not on a 16-byte boundary, take the element loop
// (the CTAs behind the tile CTAs).
constexpr int kActionTilesPerCta = 4;  // all four loads are issued up front: 43 KB in flight per CTA, five CTAs per SM
__global__ void __launch_bounds__(256) k_apply_action(const __grid_constant__ AsParams P, Workspace ws,
                                                      const float* __restrict__ actions, int64_t stride,
                                                      float* __restrict__ efforts, int64_t num_envs, int tiles,
                                                      int tile_blocks, int tail_blocks) {
  __shared__ __align__(128) float s_act[kActionTilesPerCta][kTile * kJ];
  __shared__ float s_gain[kActionTilesPerCta][kTile];
  __shared__ float s_gear[kJ];
  __shared__ uint64_t mbar[kActionTilesPerCta];
  const uint2* __restrict__ st = ws.state[ws.ctrl->parity];
  const int pending = static_cast<int>(ws.ctrl->promote_cur);
  const int tid = threadIdx.x;
  if (static_cast<int>(blockIdx.x) < tile_blocks) {
    constexpr uint32_t kBytes = kTile * kJ * 4;
    const int tile0 = blockIdx.x * kActionTilesPerCta;
    const int n_sub = min(kActionTilesPerCta, tiles - tile0);
    const int64_t env0 = static_cast<int64_t>(tile0) * kTile;
    if (tid == 0) {
      for (int k = 0; k < n_sub; ++k) {
        const uint32_t bar = smem_u32(&mbar[k]);
        mbar_init(bar, 1);
        mbar_arrive_expect_tx(bar, kBytes);
        bulk_g2s(smem_u32(s_act[k]), actions + (env0 + k * kTile) * kJ, kBytes, bar);
      }
    }
    for (int i = tid; i < n_sub * kTile; i += blockDim.x)
      (&s_gain[0][0])[i] = P.applied_gain[min(state_level(st[env0 + i].x) + pending, P.max_level)];
    if (tid < kJ) s_gear[tid] = P.joint_gears[tid];
    __syncthreads();
    for (int k = 0; k < n_sub; ++k) {
      mbar_wait(smem_u32(&mbar[k]), 0);
      for (int i = tid; i < kTile * kJ; i += blockDim.x) {
        const int e = i / kJ, j = i - e * kJ;
        s_act[k][i] = (s_gain[k][e] * s_gear[j]) * clamp_nan(s_act[k][i], -1.0f, 1.0f);
      }
      fence_proxy_async_smem();
      __syncthreads();
      if (tid == 0) {
        bulk_s2g(efforts + (env0 + k * kTile) * kJ, smem_u32(s_act[k]), kBytes);
        bulk_commit();
      }
    }
    if (tid == 0) bulk_wait_read_all();
    return;
  }
  const int64_t first = static_cast<int64_t>(tiles) * kTile * kJ;
  const int64_t total = num_envs * kJ;
  for (int64_t i = first + static_cast<int64_t>(blockIdx.x - tile_blocks) * blockDim.x + tid; i < total;
       i += static_cast<int64_t>(tail_blocks) * blockDim.x) {
    const int64_t e = i / kJ;
    const int j = static_cast<int>(i - e * kJ);
    const int level = min(state_level(st[e].x) + pending, P.max_level);
    const float act = clamp_nan(actions[e * stride + j], -1.0f, 1.0f);
    efforts[i] = (P.applied_gain[level] * P.joint_gears[j]) * act;
  }
}

struct MirrorTable {
  int32_t src[AS_OBS_DIM];
  float sign[AS_OBS_DIM];
  int32_t dim;
};

// ENV:570-660: rows [0,R) copy, rows [R,2R) = +-in[r][src[c]].  The sign is applied as a NEGATION (`-x`, what
// ENV:593,634 do), not as a product with -1: the two differ in the bits they give a NaN.
//
// A pure copy: every input element is read once and written twice.  Full tiles of kMirrorRows rows travel through
// shared memory with three TMA bulk copies -- rows in, the same buffer straight out again as the upper half, and the
// permuted / negated tile as the lower half -- so that neither half costs a second global read or a scattered access.
// The rows behind the last full tile, and tensors whose rows do not sit on 16-byte boundaries, take the element loop.
constexpr int kMirrorRows = 128;
constexpr int kMirrorSmemBytes = 2 * kMirrorRows * AS_OBS_DIM * 4;

// rows [row0, rows) of the job, element by element
__device__ __forceinline__ void mirror_rows_body(const MirrorTable& t, const float* __restrict__ in,
                                                 float* __restrict__ out, int64_t rows, int64_t row0, int block,
                                                 int n_blocks) {
  const int64_t total = rows * t.dim;
  for (int64_t i = row0 * t.dim + static_cast<int64_t>(block) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(n_blocks) * blockDim.x) {
    const int64_t r = i / t.dim;
    const int c = static_cast<int>(i - r * t.dim);
    out[i] = in[i];
    const float v = in[r * t.dim + t.src[c]];
    out[total + i] = t.sign[c] < 0.0f ? -v : v;
  }
}

template <int DIM>
__device__ __forceinline__ void mirror_tile(const MirrorTable& t, const float* __restrict__ in, float* __restrict__ out,
                                            int64_t rows, int64_t tile, unsigned char* smem, uint64_t* mbar,
                                            int* s_src) {
  constexpr uint32_t kBytes = kMirrorRows * DIM * 4;  // (a multiple of 16 for both row widths)
  float* a = reinterpret_cast<float*>(smem);
  float* b = reinterpret_cast<float*>(smem + kBytes);
  const int tid = threadIdx.x;
  const int64_t off = tile * kMirrorRows * DIM;
  const uint32_t bar = smem_u32(mbar);
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_arrive_expect_tx(bar, kBytes);
    bulk_g2s(smem_u32(a), in + off, kBytes, bar);
  }
  // (source column, with the sign in the top bit) out of the constant bank, where a warp's 32 different columns would
  // be 32 serialised reads
  if (tid < DIM) s_src[tid] = t.src[tid] | (t.sign[tid] < 0.0f ? (1 << 30) : 0);
  __syncthreads();
  mbar_wait(bar, 0);
  if (tid == 0) {  // upper half: the rows as they came
    bulk_s2g(out + off, smem_u32(a), kBytes);
    bulk_commit();
  }
  for (int i = tid; i < kMirrorRows * DIM; i += blockDim.x) {
    const int r = i / DIM, c = i - r * DIM;
    const int sc = s_src[c];
    const float v = a[r * DIM + (sc & 0xffff)];
    b[i] = (sc >> 30) ? -v : v;
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (tid == 0) {  // lower half: the mirrored rows
    bulk_s2g(out + rows * DIM + off, smem_u32(b), kBytes);
    bulk_commit();
    bulk_wait_read_all();
  }
}

struct MirrorJobs {
  const float* in[4];
  float* out[4];
  int64_t rows[4];
  int32_t kind[4];   // 0 observations (dim 59), 1 actions / mus (dim 21)
  int32_t tiles[4];  // full tiles that go through shared memory (0: the whole job takes the element loop)
  int32_t n;
};
// The tensors A2CAgentSymmetry.play_steps mirrors (obses, actions, mus: learning/a2c_ppo_mirroring.py:32-34) in ONE
// launch: blockIdx.y picks the job; blockIdx.x < tiles: one tile; the CTAs behind share the remaining rows.
__global__ void __launch_bounds__(256) k_mirror_batch(const __grid_constant__ MirrorTable t_obs,
                                                      const __grid_constant__ MirrorTable t_act,
                                                      const __grid_constant__ MirrorJobs jobs, int tail_blocks) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t mbar;
  __shared__ int s_src[AS_OBS_DIM];
  const int j = blockIdx.y;
  if (j >= jobs.n) return;
  const MirrorTable& t = jobs.kind[j] == 0 ? t_obs : t_act;
  const int tiles = jobs.tiles[j];
  const int blk = blockIdx.x;
  if (blk < tiles) {
    if (jobs.kind[j] == 0) mirror_tile<AS_OBS_DIM>(t, jobs.in[j], jobs.out[j], jobs.rows[j], blk, smem, &mbar, s_src);
    else mirror_tile<AS_NUM_JOINTS>(t, jobs.in[j], jobs.out[j], jobs.rows[j], blk, smem, &mbar, s_src);
  } else if (blk < tiles + tail_blocks) {
    mirror_rows_body(t, jobs.in[j], jobs.out[j], jobs.rows[j], static_cast<int64_t>(tiles) * kMirrorRows, blk - tiles,
                     tail_blocks);
  }
}

__global__ void __launch_bounds__(256) k_export(const __grid_constant__ AsParams P, Workspace ws, AsMdpState dst,
                                                int64_t num_envs) {
  const uint2* st = ws.state[ws.ctrl->parity];
  const int pending = static_cast<int>(ws.ctrl->promote_cur);
  const int S = static_cast<int>(P.num_steps);
  for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < num_envs;
       e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const uint2 sw = st[e];
    if (dst.curr_target_index) dst.curr_target_index[e] = state_idx(sw.x);
    if (dst.swing_leg) dst.swing_leg[e] = state_leg(sw.x);
    if (dst.target_reach_count) dst.target_reach_count[e] = state_count(sw.x);
    if (dst.episode_length) dst.episode_length[e] = state_ep(sw.x);
    if (dst.curriculum) dst.curriculum[e] = min(state_level(sw.x) + pending, P.max_level);
    if (dst.potentials) dst.potentials[e] = __uint_as_float(sw.y);
    if (dst.steps_pos || dst.steps_dphi) {
      for (int s = 0; s < S; ++s) {
        const float4 v = ws.stones[e * S + s];
        if (dst.steps_pos) {
          dst.steps_pos[(e * S + s) * 3 + 0] = v.x;
          dst.steps_pos[(e * S + s) * 3 + 1] = v.y;
          dst.steps_pos[(e * S + s) * 3 + 2] = v.z;
        }
        if (dst.steps_dphi) dst.steps_dphi[e * S + s] = v.w;
      }
    }
  }
}

__global__ void __launch_bounds__(256) k_import(const __grid_constant__ AsParams P, Workspace ws, AsMdpState src,
                                                int64_t num_envs) {
  uint2* st = ws.state[ws.ctrl->parity];
  const int pending = static_cast<int>(ws.ctrl->promote_cur);
  const int S = static_cast<int>(P.num_steps);
  for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < num_envs;
       e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    uint2 sw = st[e];
    int idx = state_idx(sw.x), leg = state_leg(sw.x), cnt = state_count(sw.x), lvl = state_level(sw.x),
        ep = state_ep(sw.x);
    if (src.curr_target_index) idx = static_cast<int>(min(max(src.curr_target_index[e], (int64_t)0), (int64_t)(S - 1)));
    if (src.swing_leg) leg = static_cast<int>(src.swing_leg[e] & 1);
    if (src.target_reach_count) cnt = static_cast<int>(min(max(src.target_reach_count[e], (int64_t)0), (int64_t)3));
    if (src.episode_length) ep = static_cast<int>(min(max(src.episode_length[e], (int64_t)0), (int64_t)kMaxEpisodeLength));
    if (src.curriculum) lvl = static_cast<int>(min(max(src.curriculum[e], (int64_t)0), (int64_t)P.max_level));
    else lvl = min(lvl + pending, P.max_level);  // a pending promotion is folded in, the flag is cleared below
    sw.x = pack_state(idx, leg, cnt, lvl, ep);
    if (src.potentials) sw.y = __float_as_uint(src.potentials[e]);
    st[e] = sw;
    if (src.steps_pos || src.steps_dphi) {
      for (int s = 0; s < S; ++s) {
        float4 v = ws.stones[e * S + s];
        if (src.steps_pos) {
          v.x = src.steps_pos[(e * S + s) * 3 + 0];
          v.y = src.steps_pos[(e * S + s) * 3 + 1];
          v.z = src.steps_pos[(e * S + s) * 3 + 2];
        }
        if (src.steps_dphi) v.w = src.steps_dphi[e * S + s];
        ws.stones[e * S + s] = v;
      }
    }
    for (int k = 0; k < 4; ++k) {  // index and/or stones may have changed: rebuild the window
      float4 v = ws.stones[e * S + window_slot_stone(idx, k, S)];
      if (k == 0) v.w = __int_as_float(idx);
      ws.window[e * 4 + k] = v;
    }
    // ... of every env, so no record is stale any more (a warp's 32 consecutive envs share one word of the bit mask)
    if ((e & 31) == 0) ws.win_stale[e >> 5] = 0u;
  }
}

// Stone poses of the listed envs in PhysX' object-major (S*N,7) x,y,z,w layout plus the matching view indices
// (rigid_object_collection.py:295-301,650-659,675).  One thread per (stone, listed env): consecutive threads write
// consecutive 28-byte rows when the ids are consecutive.
__global__ void __launch_bounds__(256) k_export_stone_poses(Workspace ws, const int32_t* __restrict__ env_ids,
                                                            int64_t n_ids, int64_t num_envs, int S,
                                                            float* __restrict__ view_poses,
                                                            int32_t* __restrict__ view_ids) {
  const int64_t total = n_ids * S;
  for (int64_t w = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; w < total;
       w += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t s = w / n_ids;
    const int64_t i = w - s * n_ids;
    const int64_t e = env_ids ? env_ids[i] : i;
    const float4 v = ws.stones[e * S + s];
    const int64_t row = s * num_envs + e;
    float* dst = view_poses + row * 7;
    dst[0] = v.x; dst[1] = v.y; dst[2] = v.z;
    dst[3] = 0.0f; dst[4] = 0.0f; dst[5] = 0.0f; dst[6] = 1.0f;  // identity, x,y,z,w
    if (view_ids) view_ids[w] = static_cast<int32_t>(row);
  }
}

// bins / histograms in and out (tests, checkpoints)
__global__ void __launch_bounds__(256) k_grid_state(Workspace ws, uint8_t* bins_dst, const uint8_t* bins_src,
                                                    unsigned int* hist_dst, const unsigned int* hist_src,
                                                    int64_t num_envs) {
  const int64_t i0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (int64_t e = i0; e < num_envs; e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    if (bins_src) ws.bin[e] = bins_src[e];
    if (bins_dst) bins_dst[e] = ws.bin[e];
  }
  if (i0 < kMaxGridBins) {
    if (hist_src) {
      ws.ctrl->grid_attempts[i0] = hist_src[i0];
      ws.ctrl->grid_successes[i0] = hist_src[kMaxGridBins + i0];
    }
    if (hist_dst) {
      hist_dst[i0] = ws.ctrl->grid_attempts[i0];
      hist_dst[kMaxGridBins + i0] = ws.ctrl->grid_successes[i0];
    }
  }
}

// ------------------------------------------------------------------------------------------------ 3-call path, pass 2
// as_step_pass1 ran pass 2 speculatively for every env that did not reset (state in the other buffer, observation
// rows final).  What is left of ENV:567 when some env did reset:
//   k_pass2_commit   one warp per env that reset: `_compute_useful_values` + its observation row from the physics
//                    state as it is AFTER the PhysX writes of ENV:563-565 (general orientation, the body positions the
//                    simulator reports now, the contact rows scene.reset zeroed), into the other state buffer; the
//                    last CTA then makes that buffer the current one.
// and when none did (DRL:360 skips `_reset_idx`):
//   k_pass2_revert   the observation tails of pass 1 back into the observation rows; the state buffer of pass 1 stays.
struct CommitArgs {
  AsParams P;
  JointConsts jc;
  AsStateIn in;     // the views as they are after the writes
  Workspace ws;
  float* obs;       // (N,59)
  float obs_clip;
  float inv_step_dt;
  int64_t num_envs;
  int32_t revert_if_none;  // device-side reset list: whether any env reset is only known here -- none did: behave as
                           // k_pass2_revert (DRL:360 would have skipped `_reset_idx`)
  int32_t peer_three_call; // global 3-call mode: "none did" means none on ANY shard (Ctrl::any_reset), and this step's
                           // grid outcomes stay in Ctrl::grid_delta_* for the next k_peer_exchange to sum and add
};

// Takes the speculated pass 2 back (grid-stride over the whole launch): the observation tails of pass 1 return to the
// observation rows, and the pass-2 advances pass 1 counted leave the statistics.  The state buffer of pass 1 stays.
__device__ __forceinline__ void revert_pass2(const Workspace& ws, float* __restrict__ obs, float obs_clip,
                                             int64_t num_envs) {
  const int64_t total = num_envs * 11;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t e = i / 11;
    const int c = static_cast<int>(i - e * 11);
    obs[e * kObs + 48 + c] = clip_obs(reinterpret_cast<const float*>(ws.tail1 + e * 3)[c], obs_clip);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) ws.ctrl->stats.n_advanced -= ws.ctrl->last_adv2;
}

__global__ void __launch_bounds__(256) k_pass2_commit(const __grid_constant__ CommitArgs a) {
  __shared__ float s_row[8][4][20];
  const AsParams& P = a.P;
  Ctrl* ctrl = a.ws.ctrl;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t n = ctrl->n_reset_list;
  if (n == 0 && a.revert_if_none && !(a.peer_three_call && ctrl->any_reset)) {
    revert_pass2(a.ws, a.obs, a.obs_clip, a.num_envs);
    return;
  }
  uint2* st = a.ws.state[ctrl->parity ^ 1u];  // the buffer pass 1 speculated into and as_reset wrote
  const bool exact = a.jc.exact_div != 0;
  const AsStateIn& in = a.in;
  // four envs per warp, eight lanes each (see k_reset_rows: independent load chains per warp)
  const int grp = lane >> 3, g = lane & 7;
  for (int64_t w0 = warp * 4; w0 < n; w0 += n_warps * 4) {
    const int64_t w = w0 + grp;
    const bool have = w < n;
    int64_t e = 0;
    if (have) {
      e = a.ws.reset_ids[w];
      const uint2 sw = st[e];
      Mdp m{state_idx(sw.x), state_leg(sw.x), state_count(sw.x), __uint_as_float(sw.y)};
      const int level = state_level(sw.x), ep = state_ep(sw.x);
      // every lane of the group computes the env's scalars (same addresses: broadcast loads)
      const float* rp = in.root_pos + e * in.root_pos_stride;
      const float* rq = in.root_quat + e * in.root_quat_stride;
      const float* rv = in.root_lin_vel + e * in.root_lin_vel_stride;
      const Vec3 p{rp[0], rp[1], rp[2]}, v{rv[0], rv[1], rv[2]};
      const Quat q = in.quat_xyzw ? Quat{rq[3], rq[0], rq[1], rq[2]} : Quat{rq[0], rq[1], rq[2], rq[3]};
      const float* body = in.body_pos + e * in.body_env_stride;
      const float* b_r = body + in.right_foot_row * in.body_row_stride;
      const float* b_l = body + in.left_foot_row * in.body_row_stride;
      const float* b_t = body + in.torso_row * in.body_row_stride;
      const Vec3 rf{b_r[0], b_r[1], b_r[2]}, lf{b_l[0], b_l[1], b_l[2]};
      const int S = static_cast<int>(P.num_steps);
      const float4* stones = a.ws.stones + e * S;
      float4 s_prev = stones[window_slot_stone(m.idx, 0, S)], s_curr = stones[window_slot_stone(m.idx, 1, S)],
             s_next = stones[window_slot_stone(m.idx, 2, S)];
      const float f_r = contact_norm(in.contact_right + e * in.contact_right_stride, m.idx, false);
      const float f_l = contact_norm(in.contact_left + e * in.contact_left_stride, m.idx, false);
      const float h = b_t[2] - min_nan(lf.z, rf.z);                       // ENV:281-283
      float roll, pitch;
      euler_roll_pitch(q, roll, pitch);                                    // ENV:285
      const Vec3 vb = rotate_by_inverse(q, v);                             // ENV:293
      const Quat inv = quat_inverse(q);
      PassOut po{};
      const FootGeom gm = foot_geometry(P, rf, lf, f_r > P.contact_epsilon, f_l > P.contact_epsilon, s_curr);
      if (foot_update(P, gm, m, po, S)) {  // (cannot happen on zeroed contact rows; kept general)
        s_prev = s_curr;
        s_curr = s_next;
        s_next = stones[min(m.idx + 1, S - 1)];
      }
      targets_and_potential(P, a.inv_step_dt, exact, p, inv, s_prev, s_curr, s_next, m, po);
      if (g == 0) {
        uint2 out;
        out.x = pack_state(m.idx, m.leg, m.count, level, ep);
        out.y = __float_as_uint(m.pot);
        st[e] = out;
        atomicOr(&a.ws.win_stale[e >> 5], 1u << (e & 31));  // its stone window is for k_prepare* to refresh
        float* r = s_row[wib][grp];
        r[0] = h; r[1] = roll; r[2] = pitch; r[3] = vb.x; r[4] = vb.y; r[5] = vb.z;
        r[6] = po.contact_r; r[7] = po.contact_l;
        r[8] = po.tb0.x; r[9] = po.tb0.y; r[10] = po.tb0.z; r[11] = po.tb1.x; r[12] = po.tb1.y; r[13] = po.tb1.z;
        r[14] = po.tb2.x; r[15] = po.tb2.y; r[16] = po.tb2.z;
      }
    }
    __syncwarp();
    if (have) {
      float* row = a.obs + e * kObs;
      for (int c = g; c < 17; c += 8)   // ENV:332-335 (columns 0..5) and ENV:338-339 (columns 48..58)
        row[c < 6 ? c : 48 + c - 6] = clip_obs(s_row[wib][grp][c], a.obs_clip);
      for (int j = g; j < kJ; j += 8) {
        const float jp = in.joint_pos[e * in.joint_pos_stride + j];
        const float jv = in.joint_vel[e * in.joint_vel_stride + j];
        row[6 + j] = clip_obs(scale_joint(a.jc.c[j], jp, exact), a.obs_clip);                     // ENV:336
        row[6 + kJ + j] = clip_obs(clamp_nan(jv * P.dof_vel_scale, -5.0f, 5.0f), a.obs_clip);     // ENV:337
      }
    }
    __syncwarp();
  }
  // the last CTA makes the speculated buffer the current state
  __shared__ unsigned int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(&ctrl->blocks_done2, 1u) == gridDim.x - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (s_last && (P.flags & AS_FLAG_GRID_CURRICULUM) && !a.peer_three_call) {
    // this step's episode outcomes (k_reset_rows) join the difficulty-grid histograms of this shard, as the fused
    // step's finish does
    for (int i = threadIdx.x; i < kMaxGridBins; i += blockDim.x) {
      grid_fold(ctrl->grid_attempts[i], ctrl->grid_successes[i], ctrl->grid_delta_att[i], ctrl->grid_delta_succ[i]);
      ctrl->grid_delta_att[i] = ctrl->grid_delta_succ[i] = 0u;
    }
  }
  if (s_last && threadIdx.x == 0) {
    ctrl->parity ^= 1u;
    ctrl->n_reset_list = 0;
    ctrl->n_regen_list = 0;
    ctrl->blocks_done2 = 0;
  }
}

// peer_three_call: global 3-call mode.  When an env of another shard reset, the reference runs pass 2 for every env
// (DRL:359-360 and ENV:567 look at all envs): keep what pass 1 speculated -- observations, state buffer, advances.
__global__ void __launch_bounds__(256) k_pass2_revert(Workspace ws, float* __restrict__ obs, float obs_clip,
                                                      int64_t num_envs, int32_t peer_three_call) {
  const bool commit = peer_three_call && ws.ctrl->any_reset;
  if (!commit) revert_pass2(ws, obs, obs_clip, num_envs);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ws.ctrl->n_reset_list = 0;
    if (commit) ws.ctrl->parity ^= 1u;  // the speculated buffer becomes the current state
  }
}

// `_reset_idx` called outside a step (as_reset without a preceding as_step_pass1): the numerator of ENV:471 from the
// state words as they are, and a fresh Philox step counter for the draws of this reset.  One CTA.
__global__ void __launch_bounds__(1024) k_prepare_reset(Workspace ws, int64_t num_envs) {
  __shared__ unsigned long long s_sum[32];
  Ctrl* ctrl = ws.ctrl;
  const uint2* st = ws.state[ctrl->parity];
  unsigned long long sum = 0;
  for (int64_t e = threadIdx.x; e < num_envs; e += blockDim.x) sum += static_cast<unsigned long long>(state_idx(st[e].x));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(kFullMask, sum, o);
  if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long tot = 0;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) tot += s_sum[w];
    ctrl->stats.n_envs = num_envs;
    ctrl->stats.sum_target_index = static_cast<int64_t>(tot);
    ctrl->step_counter += 1ull;
    ctrl->stats.step_counter = static_cast<int64_t>(ctrl->step_counter);
  }
}

// as_restore: the fields of a saved control block that are MDP state (parity of the state buffers, pending promotion,
// Philox step counter, folded statistics, difficulty-grid histograms and the grid outcomes the global 3-call mode keeps
// pending between steps -- zero between steps in every other mode).  Live bookkeeping stays: the peer-exchange epoch
// (the peers' slots hold flags of the live epoch), diagnostics counters.
__global__ void k_restore_ctrl(Ctrl* ctrl, const Ctrl* saved) {
  const int t = threadIdx.x;
  if (t == 0) {
    ctrl->parity = saved->parity;
    ctrl->promote_cur = saved->promote_cur;
    ctrl->step_counter = saved->step_counter;
    ctrl->stats = saved->stats;
    ctrl->gx.stats = saved->gx.stats;
    ctrl->last_adv2 = saved->last_adv2;
    ctrl->stats_folded = 0;
    ctrl->blocks_done = ctrl->blocks_done2 = 0;
    ctrl->n_reset_list = ctrl->n_regen_list = 0;
  }
  for (int i = t; i < kMaxGridBins; i += blockDim.x) {
    ctrl->grid_attempts[i] = saved->grid_attempts[i];
    ctrl->grid_successes[i] = saved->grid_successes[i];
    ctrl->grid_delta_att[i] = saved->grid_delta_att[i];
    ctrl->grid_delta_succ[i] = saved->grid_delta_succ[i];
  }
  for (int i = t; i < kSlots * kNumCounters; i += blockDim.x) (&ctrl->slots[0][0])[i] = 0u;
  for (int i = t; i < kSlots; i += blockDim.x) ctrl->slot_reward[i] = 0.0f;
}

__global__ void k_clear_promotion(Ctrl* ctrl) {
  if (threadIdx.x == 0 && blockIdx.x == 0) ctrl->promote_cur = 0;
}

}  // namespace as
