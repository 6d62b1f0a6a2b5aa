// Kernel (a): the fused Allsteps-v0 MDP step for sm_100a.
//
// One CTA of 256 threads owns a tile of 128 consecutive envs, TWO threads per env in two warp roles (warps 0-3 "MDP
// role", warps 4-7 "joint role"; see process_tile).
//
//   HBM -> SMEM   the row-major PhysX views of the tile (joint_pos/joint_vel/actions (128,21), root pos/quat/vel,
//                 feet+torso positions) are contiguous byte ranges, so one elected thread moves each of them with a
//                 single TMA bulk copy (cp.async.bulk.shared.global, completion on an mbarrier).  A thread then
//                 reads ITS row from shared memory: row strides 21, 3, 9 are odd => bank-conflict free, and the
//                 global side is perfectly coalesced although the layout is array-of-structs.
//   gathers       the packed 8-byte MDP state word and the 64-byte stone-window record are coalesced loads; the two
//                 contact norms of the current stone come as one coalesced record from k_contact_gather* (large
//                 batches) or are gathered here (small, launch-bound batches); stones a step has to fetch out of the
//                 S x 16-byte stone rows travel global -> shared asynchronously (cp.async) when nothing waits for them.
//   compute       dones -> pass 1 -> rewards -> masked reset (Philox) -> pass 2 -> observations.  The code of both
//                 roles is kept STRAIGHT-LINE on purpose: the kernel is bound by how its two instruction streams
//                 schedule (DESIGN.md section 6), every branch ends a basic block and a taken one refetches
//                 instructions -- hence the template parameters instead of run-time choices, the branch-free sqrt /
//                 quotients of as_math.cuh, and full and ragged tiles as separate kernels.
//   SMEM -> HBM   the (128,59) observation tile is assembled in shared memory (row stride 59, odd) on top of the
//                 consumed input tiles and leaves with one TMA bulk store; reward / flags / state word are
//                 coalesced per-thread stores.
//
// Reference semantics reproduced (ENV = allsteps_env.py, DRL = direct_rl_env.py of the reference):
//   DRL:351 episode counter, ENV:276-324 pass, ENV:396-405 dones, ENV:347-394 rewards, ENV:469-567 reset + pass 2
//   for ALL envs when any env resets (SURVEY D7), ENV:326-345 observations.
#pragma once
#include <type_traits>
#include "as_internal.cuh"
#include "as_math.cuh"
#include "philox.cuh"

namespace as {

// ------------------------------------------------------------------------------------------------ SMEM plan
constexpr int kOffJp = 0;
constexpr int kOffJv = kOffJp + kTile * kJ * 4;
constexpr int kOffAct = kOffJv + kTile * kJ * 4;
constexpr int kOffRp = kOffAct + kTile * kJ * 4;
constexpr int kOffRq = kOffRp + kTile * 3 * 4;
constexpr int kOffRv = kOffRq + kTile * 4 * 4;
constexpr int kOffBody = kOffRv + kTile * 3 * 4;
constexpr int kOffOrg = kOffBody + kTile * 9 * 4;   // env origins of the tile (needed by the envs that reset)
constexpr int kOffMisc = kOffOrg + kTile * 3 * 4;
constexpr int kMiscBytes = AS_KTILE == 128 ? 8192 : 4864;
constexpr int kOffW3 = kOffMisc + kMiscBytes;     // float4 per env: the stone entering the window record (see write-back)
constexpr int kOffPhx = kOffW3 + kTile * 16;  // uint4 per joint-role lane: Philox blocks of five envs of a warp that reset
constexpr int kSmemBytes = kOffPhx + kTile * 16;
static_assert((512 / AS_KTILE) * (kSmemBytes + 1024) <= 233472 || AS_KTILE != 128, "four CTAs per SM");
// PACKED instantiations (root pos / quat / lin vel are slices of ONE (N,13) root_state_w tensor, which is what Isaac
// Lab hands out): the (kTile,13) tile is a single contiguous 16-byte aligned range and travels as one bulk copy
// into the place of the three root tiles; the body tile moves up behind it and the env-origin tile to the very end.
constexpr int kRootRow = AS_ROOT_STATE_DIM;  // 13 floats: pos 0..2, quat 3..6, lin vel 7..9, ang vel 10..12
constexpr int kOffBodyPacked = kOffRp + kTile * kRootRow * 4;
constexpr int kOffOrgPacked = kSmemBytes;
constexpr int kSmemBytesPacked = kSmemBytes + kTile * 3 * 4;
static_assert(kOffBodyPacked + kTile * 9 * 4 <= kOffMisc && kOffBodyPacked % 16 == 0 && kOffOrgPacked % 16 == 0, "packed layout");
static_assert((512 / AS_KTILE) * (kSmemBytesPacked + 1024) <= 233472 || AS_KTILE != 128, "four CTAs per SM (packed)");
static_assert(kTile * kObs * 4 <= kOffRp, "observation tile must fit over the joint/action tiles it aliases");
static_assert(kOffJv % 16 == 0 && kOffAct % 16 == 0 && kOffRp % 16 == 0 && kOffRq % 16 == 0 &&
                  kOffRv % 16 == 0 && kOffBody % 16 == 0 && kOffOrg % 16 == 0 && kOffMisc % 16 == 0,
              "bulk copies need 16-byte aligned shared addresses");

// Per-joint tables of the reset pose, one entry per lane.  Lane-indexed reads of kernel parameters would go
// through the constant bank, which serialises divergent addresses; shared memory / registers do not.
struct ResetTables {
  float4 jc[32];  // JointConsts record of joint `lane`
  float pose[32], pose_mirrored[32], vel_mirrored[32];
};

constexpr int kThreads = 2 * kTile;  // two threads per env: one MDP-role and one joint-role warp per 32 envs

struct Misc {  // lives at kOffMisc, never aliased
  unsigned long long mbar_root;   // completion of the root / body tiles
  unsigned long long mbar_joint;  // completion of the joint_pos / joint_vel / actions tiles
  unsigned int wcnt[kTile / 32][kNumCounters];  // per-warp step counters
  float wreward[kTile / 32];
  unsigned int is_last;
  ResetTables rt;
  // exchanged between the two roles at the CTA barrier
  float red_energy[kTile];   // sum_j |joint_vel * action|, ENV:365
  float red_actsq[kTile];    // sum_j action^2, ENV:364
  int red_limit[kTile];      // count_j |joint_pos_scaled| > 0.99, ENV:367
  unsigned int flags[kTile]; // bit 0: env resets this step
  unsigned char coin[kTile]; // the mirror coin of ENV:518 for this step (used only if the env resets)
  // orientation results computed by the joint role from the root tile while its own tiles are in flight
  float x_roll[kTile], x_pitch[kTile];
  float x_vb[3][kTile];      // root velocity in the root frame, parked here across the joint loop (registers are short)
  float x_inv[4][kTile];     // quat_inv(root_quat), MATH:238-248
};
static_assert(sizeof(Misc) <= kMiscBytes, "misc block");

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!ok);
}
// TMA 1-D bulk copy global -> shared, completion counted in bytes on the mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// TMA 1-D bulk copy shared -> global.
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// Named barrier 1: the joint role arrives when the orientation results are in shared memory, the MDP role waits for
// them just before it needs them (barrier 0 is __syncthreads).
__device__ __forceinline__ void orient_arrive() { asm volatile("bar.arrive 1, %0;" ::"n"(2 * kTile) : "memory"); }
__device__ __forceinline__ void orient_wait() { asm volatile("bar.sync 1, %0;" ::"n"(2 * kTile) : "memory"); }
// Named barrier 2: reset flags, MDP role (producer, early) -> joint role (consumer).
__device__ __forceinline__ void flags_arrive() { asm volatile("bar.arrive 2, %0;" ::"n"(2 * kTile) : "memory"); }
__device__ __forceinline__ void flags_wait() { asm volatile("bar.sync 2, %0;" ::"n"(2 * kTile) : "memory"); }
// Named barrier 3: the joint-role warps among themselves -- every joint/action row has been consumed, the observation
// tile may overwrite them.
__device__ __forceinline__ void joint_rows_consumed() { asm volatile("bar.sync 3, %0;" ::"n"(kTile) : "memory"); }
// Named barrier 4: "rows consumed + reward sums written", joint role (producer) -> MDP role (consumer).
__device__ __forceinline__ void sums_arrive() { asm volatile("bar.arrive 4, %0;" ::"n"(2 * kTile) : "memory"); }
__device__ __forceinline__ void sums_wait() { asm volatile("bar.sync 4, %0;" ::"n"(2 * kTile) : "memory"); }
// Asynchronous 16-byte copy global -> shared (LDGSTS): the issuing thread does not wait for the data.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global.L2::64B [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// ------------------------------------------------------------------------------------------------ staging
// A tile of an (N,W) view can be moved by the bulk-copy engine when the view is dense (stride == W), the tile starts
// on a 16-byte boundary and its byte count is a multiple of 16.  The first two are properties of the view: the
// host evaluates them once per launch (StepArgs::dense16, one bit per array; every tile starts on a multiple of
// 128 rows, and 128 * W * 4 is a multiple of 16 for every W); only the ragged last tile needs the third.
enum DenseBit { kDenseJp = 1, kDenseJv = 2, kDenseAct = 4, kDenseRp = 8, kDenseRq = 16, kDenseRv = 32, kDenseBody = 64,
                kDenseOrg = 128, kDenseObs = 256 };
template <int W>
__device__ __forceinline__ bool bulk_ok(uint32_t dense16, uint32_t bit, int n_valid) {
  return (dense16 & bit) && (((n_valid * W) & 3) == 0);
}
// All arrays at once: a full tile keeps every dense bit; a ragged tile keeps those whose byte count is a multiple of 16.
__device__ __forceinline__ uint32_t bulk_mask(uint32_t dense16, int n_valid) {
  if (n_valid == kTile) return dense16;
  uint32_t m = dense16 & (kDenseRq);  // 16-byte rows always qualify
  if ((n_valid & 3) == 0) m = dense16;  // every other row width (84, 12, 36, 236 bytes) needs a multiple of 4 rows
  return m;
}
template <int W>
__device__ __forceinline__ void coop_load(float* dst, const float* base, int64_t stride, int64_t env0, int n_valid) {
  for (int i = threadIdx.x; i < n_valid * W; i += 2 * kTile) {
    const int r = i / W;
    const int c = i - r * W;
    dst[i] = __ldg(base + (env0 + r) * stride + c);
  }
}

// Scattered reads (one 12/16-byte item out of a 12 S / 16 S-byte row per env, 240 / 320 bytes at the default S = 20):
// by default a miss makes L2 pull the whole 128-byte line out of DRAM; the L2::64B qualifier limits the fill to the
// 64-byte half that holds the item.  These gathers are DRAM-byte bound, so that halves their cost
// (tools/gather_probe.cu: 259 -> 143 DRAM bytes per env, 44 -> 27 us per 1M envs).  SASS: LDG.E.LTC64B...CONSTANT.
__device__ __forceinline__ float4 ldg64_f4(const float4* p) {
  float4 r;
  asm("ld.global.nc.L2::64B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
// The same for data that is read exactly once (the contact matrices): the lines are also marked "evict first" in L2, so
// that the gather's fills do not push out what the step kernel is about to read (state words, contact records, stone
// windows written / touched by the same kernel).  Measured at 1 M envs (profiles/r02_experiments.txt): no hints 188.5 us
// per step; this + "evict last" on the contact record 185.3; + "evict last" on the step kernel's state-word store (the
// next k_prepare* reads it first thing) 184.0-184.4.  "Evict last" on the window refresh helps at 262 144 envs (62.5
// against 64.3) and costs at 1 M (187.7): the refresh stores without a hint.
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ldg64_once_f4(const float4* p, uint64_t pol) {
  float4 r;
  asm("ld.global.nc.L2::cache_hint.L2::64B.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
      : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void st_keep_u8(uint8_t* p, unsigned v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u8 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep_u2(uint2* p, const uint2& v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v2.u32 [%0], {%1,%2}, %3;" ::"l"(p), "r"(v.x), "r"(v.y), "l"(pol) : "memory");
}
__device__ __forceinline__ float ldg64_f(const float* p) {
  float r;
  asm("ld.global.nc.L2::64B.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

// Norm of the 12-byte contact-force vector of stone `idx` inside one env's (S,3) row.  When the row is 16-byte
// aligned the vector is fetched with one or two aligned 128-bit loads instead of three scalar ones: the same
// sectors, half the requests through the L1 miss path.
__device__ __forceinline__ float contact_norm(const float* row, int idx, bool aligned16) {
  float x, y, z;
  if (aligned16) {
    const int o = idx * 3;
    const int k = o & 3;
    const float4* c = reinterpret_cast<const float4*>(row) + (o >> 2);
    const float4 c0 = ldg64_f4(c);
    if (k == 0) {
      x = c0.x; y = c0.y; z = c0.z;
    } else if (k == 1) {
      x = c0.y; y = c0.z; z = c0.w;
    } else {
      const float4 c1 = ldg64_f4(c + 1);
      if (k == 2) {
        x = c0.z; y = c0.w; z = c1.x;
      } else {
        x = c0.w; y = c1.x; z = c1.y;
      }
    }
  } else {
    const float* f = row + idx * 3;
    x = ldg64_f(f); y = ldg64_f(f + 1); z = ldg64_f(f + 2);
  }
  return norm3(x, y, z);  // ENV:421-424
}

// The observation clamp of AsStepOut.obs_clip for one value (c == 0: raw).  Comparisons, not fminf/fmaxf: torch.clamp
// hands NaN through.
__device__ __forceinline__ float clip_obs(float v, float c) {
  return c > 0.0f ? (v < -c ? -c : (v > c ? c : v)) : v;
}

// ------------------------------------------------------------------------------------------------ one pass
struct Mdp {
  int idx, leg, count;
  float pot;
};
struct FootGeom {  // ENV:421-431 relative to the CURRENT stone
  bool press_r, press_l;
  float d_r, d_l;
};
struct PassOut {
  float contact_r, contact_l;  // foot_contact (right, left) as 0/1 floats, ENV:426
  float d_swing;               // foot_to_target_dist_xy[n, swing_leg] with the POST-update leg, ENV:371
  float body_dist;             // ENV:410
  float old_pot;               // ENV:415
  bool reached, advanced;
  Vec3 tb0, tb1, tb2;          // targets_b rows (prev, curr, next), ENV:302-316
};

__device__ __forceinline__ FootGeom foot_geometry(const AsParams& P, const Vec3& rf, const Vec3& lf, bool press_r,
                                                  bool press_l, const float4& s_curr) {
  FootGeom g;
  g.press_r = press_r;  // ENV:425: |F| > 1e-4 on the current stone (evaluated where the force vector is read)
  g.press_l = press_l;
  g.d_r = norm2(rf.x - s_curr.x, rf.y - s_curr.y);  // ENV:431
  g.d_l = norm2(lf.x - s_curr.x, lf.y - s_curr.y);
  return g;
}

// ENV:433-457: reach counter, leg flip, index advance.  Returns true when the index changed (window must shift).
// S: the course length.
__device__ __forceinline__ bool foot_update(const AsParams& P, const FootGeom& g, Mdp& m, PassOut& o, int S) {
  o.contact_r = g.press_r ? 1.0f : 0.0f;
  o.contact_l = g.press_l ? 1.0f : 0.0f;
  o.reached = m.leg ? (g.press_l && g.d_l < P.step_radius) : (g.press_r && g.d_r < P.step_radius);
  m.count += o.reached ? 1 : 0;
  o.advanced = m.count >= P.stop_frames;
  bool moved = false;
  if (o.advanced) {
    m.leg ^= 1;
    const int nidx = min(m.idx + 1, S - 1);
    moved = nidx != m.idx;
    m.idx = nidx;
    m.count = 0;
  }
  o.d_swing = m.leg ? g.d_l : g.d_r;
  return moved;
}

// ENV:459-467 + ENV:302-316 + ENV:407-416 for a general root orientation (`inv` = quat_inv(root_quat)).
// ENV:416 potentials = -dist / step_dt
__device__ __forceinline__ float potential_of(const AsParams& P, float inv_step_dt, float dist, bool exact) {
  return exact ? (-dist) / P.step_dt : div_by_const(-dist, P.step_dt, inv_step_dt);
}
__device__ __forceinline__ void targets_and_potential(const AsParams& P, float inv_step_dt, bool exact, const Vec3& p,
                                                      const Quat& inv, const float4& s_prev, const float4& s_curr,
                                                      const float4& s_next, Mdp& m, PassOut& o) {
  o.tb0 = point_in_frame(p, inv, Vec3{s_prev.x, s_prev.y, s_prev.z});
  o.tb1 = point_in_frame(p, inv, Vec3{s_curr.x, s_curr.y, s_curr.z});
  o.tb2 = point_in_frame(p, inv, Vec3{s_next.x, s_next.y, s_next.z});
  o.body_dist = norm2(s_next.x - p.x, s_next.y - p.y);
  o.old_pot = m.pot;
  m.pot = potential_of(P, inv_step_dt, o.body_dist, exact);
}

// First three stones of ANY generated sequence are fixed (ENV:144-150): the pass after a regeneration needs
// only these, so the step kernel does not wait for the regeneration kernel.
__device__ __forceinline__ void first_three_stones(const AsParams& P, const Vec3& origin, float4& s0, float4& s1,
                                                   float4& s2) {
  const float half_pi = 1.5707963705062866f;
  const float st = sinf(half_pi), ct = cosf(half_pi);
  const float dx = (P.init_step_separation * st) * cosf(0.0f);
  const float dy = (P.init_step_separation * st) * sinf(0.0f);
  const float dz = P.init_step_separation * ct;
  double x = 0.0, y = 0.0, z = 0.0;  // torch.cumsum on CPU accumulates fp32 inputs in double
  s0 = make_float4(static_cast<float>(x) + origin.x, static_cast<float>(y) + origin.y,
                   static_cast<float>(z) + origin.z, 0.0f);
  x += dx; y += dy; z += dz;
  s1 = make_float4(static_cast<float>(x) + origin.x, static_cast<float>(y) + origin.y,
                   static_cast<float>(z) + origin.z, 0.0f);
  x += dx; y += dy; z += dz;
  s2 = make_float4(static_cast<float>(x) + origin.x, static_cast<float>(y) + origin.y,
                   static_cast<float>(z) + origin.z, 0.0f);
}

// MATH:22-40 with the per-joint constants precomputed on the host (JointConsts): the quotient
// (2*(x - offset)) / range is produced by the two-FMA correction q = fma(fma(-q0, range, n), inv, q0), which is the
// correctly rounded quotient when inv = RN(1/range) (Markstein); as_create falls back to a true division for a
// joint whose range has an all-ones significand (the theorem's excluded case).
// `exact` (true division) is never decided per joint: the host knows whether any divisor is an excluded case and
// launches the hot instantiations (EXACT = 0) only when none is, so they have no branch for it -- every branch ends a
// basic block and, when taken, costs an instruction refetch; with one inside each of the 21 unrolled joint
// iterations the joint loop ran 2.5x slower.  The others (EXACT = 2) choose once, ahead of the joint loop.
// The factor 2 of MATH:39 is folded into the constants (c = offset, range / 2, 2 / range): scaling by a power of two is
// exact, so (2 d) / range and d / (range / 2) are the same real quotient and every rounding of the two-FMA sequence
// lands on the same value (outside the denormal range) -- one multiplication per joint less.
__device__ __forceinline__ float scale_joint(const float4& c, float x, bool exact) {
  const float d = x - c.x;
  return exact ? d / c.y : div_by_const(d, c.y, c.z);
}
// EXACT template argument of process_tile / k_step: 0 two-FMA quotients, 2 decided at run time from
// JointConsts::exact_div (the launches off the hot path, to keep the number of instantiations down).
template <int EXACT>
__device__ __forceinline__ bool use_exact_div(const JointConsts& C) {
  return EXACT == 2 && C.exact_div != 0;
}

// Start-pose joint value of a reset env (ENV:505-560): running-start pose (already mirrored or not), uniform
// noise, clip in the unit range.  `base`, `lo`, `hi` are this joint's table entries.
// (offset and range of the record are (lo + hi) * 0.5 and hi - lo with the roundings of MATH:36-40 / MATH:57-61.)
__device__ __forceinline__ float reset_joint_value(const AsParams& P, float base, const float4& c, float u, bool exact) {
  const float noisy = base + (u * P.noise_span + P.noise_lower);
  float unit = scale_joint(c, noisy, exact);
  unit = clamp_nan(unit, P.clip_lower, P.clip_upper);
  return unit * c.y + c.x;  // MATH:43-61 unscale_transform: (unit * range) * 0.5 + offset, the halving being exact
}

// The same with the joint limits themselves and a true division (k_reset_rows, off the hot path); identical results.
__device__ __forceinline__ float reset_joint_value(const AsParams& P, float base, float lo, float hi, float u) {
  const float noisy = base + (u * P.noise_span + P.noise_lower);
  float unit = scale_to_unit(noisy, lo, hi);
  unit = clamp_nan(unit, P.clip_lower, P.clip_upper);
  return unscale_from_unit(unit, lo, hi);
}
__device__ __forceinline__ void load_reset_tables(const AsParams& P, int lane, float& lo, float& hi, float& pose,
                                                  float& pose_m, float& vel_m) {
  const int j = lane < kJ ? lane : 0;
  lo = P.joint_lower[j];
  hi = P.joint_upper[j];
  pose = P.reset_pose[j];
  pose_m = P.reset_pose[P.mirror_src[j]] * P.mirror_sign[j];  // ENV:522-526
  vel_m = 0.0f * P.mirror_sign[j];                             // default_joint_vel is zero, ENV:513,528-532
}

// Fills one lane's entries of the reset tables (called once per CTA by the first warp, or kept in registers).
__device__ __forceinline__ void load_reset_tables(const AsParams& P, const JointConsts& C, int lane, float4& jc,
                                                  float& pose, float& pose_m, float& vel_m) {
  const int j = lane < kJ ? lane : 0;
  jc = C.c[j];
  pose = P.reset_pose[j];
  pose_m = P.reset_pose[P.mirror_src[j]] * P.mirror_sign[j];  // ENV:522-526
  vel_m = 0.0f * P.mirror_sign[j];                             // default_joint_vel is zero, ENV:513,528-532
}

// ------------------------------------------------------------------------------------------------ statistics
// Sum of one per-step counter over the replicated slots (any warp may call; all 32 lanes participate).
__device__ __forceinline__ unsigned slot_sum(const Ctrl* ctrl, int which) {
  const unsigned v = __ldcg(&ctrl->slots[threadIdx.x & 31][which]);
  return __reduce_add_sync(0xffffffffu, v);
}

// Folds the slots into ctrl->stats and clears them: one warp, one lane per slot, lane 0 writes the totals.  Nobody may
// still be adding to the slots (the caller is the last CTA of the step kernel, or a kernel behind it in stream order),
// so plain L2 loads followed by independent zeroing stores do: one memory round trip for the whole fold.  Returns the
// step's reset count in every lane.
__device__ __forceinline__ unsigned fold_stats_warp(Ctrl* ctrl, int64_t num_envs, int lane) {
  unsigned tot[kNumCounters];
#pragma unroll
  for (int c = 0; c < kNumCounters; ++c) {
    const unsigned v = __ldcg(&ctrl->slots[lane][c]);
    __stcg(&ctrl->slots[lane][c], 0u);
    tot[c] = c == kCntLevelMax ? __reduce_max_sync(0xffffffffu, v) : __reduce_add_sync(0xffffffffu, v);
  }
  float rsum = __ldcg(&ctrl->slot_reward[lane]);
  __stcg(&ctrl->slot_reward[lane], 0.0f);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rsum += __shfl_xor_sync(0xffffffffu, rsum, o);
  if (lane == 0) {
    AsStats& st = ctrl->stats;
    st.n_envs = num_envs;
    st.n_reset = tot[kCntReset];
    st.n_terminated = tot[kCntTerminated];
    st.n_time_out = tot[kCntTimeOut];
    st.n_fell = tot[kCntFell];
    st.n_so_fast = tot[kCntSoFast];
    st.n_died = tot[kCntDied];
    st.n_advanced = static_cast<int64_t>(tot[kCntAdvanced1]) + tot[kCntAdvanced2];
    st.sum_target_index = tot[kCntSumIndex];
    st.n_regenerated = tot[kCntRegen];
    st.level = tot[kCntLevelMax];
    st.step_counter = static_cast<int64_t>(ctrl->step_counter);
    st.sum_reward = static_cast<double>(rsum);
    st.n_missed = tot[kCntMissed];
    ctrl->last_adv2 = tot[kCntAdvanced2];
  }
  return tot[kCntReset];
}

// ENV:471-472 promotion rule on step statistics (this shard's, or summed over ranks).
__device__ __forceinline__ uint32_t promotion_rule(const AsParams& P, int64_t n_reset, int64_t sum_index,
                                                   int64_t n_envs) {
  if (n_reset <= 0 || n_envs <= 0) return 0u;  // `_reset_idx` is only entered when an env resets, DRL:360
  const float mean = static_cast<float>(sum_index) / static_cast<float>(n_envs);
  return mean > P.progress_threshold ? 1u : 0u;
}
__device__ __forceinline__ uint32_t promotion_decision(const AsParams& P, const AsStats& s) {
  return promotion_rule(P, s.n_reset, s.sum_target_index, s.n_envs);
}

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// The cross-shard sum of the ten step counters by ONE warp (lane r talks to rank r): store this shard's counters into
// OUR slot of rank r's buffer, then the epoch as the flag (release); poll rank r's slot in OUR buffer for the same epoch
// (acquire) and read its counters; sum over the lanes.  Returns the number of peers that did not deliver in time.
// Two slots per sender (epoch parity): a rank can run at most one step ahead of a peer that has not yet read, because it
// cannot close step t+1 without that peer's step-t+1 counters.
__device__ __forceinline__ unsigned peer_sum_counters_warp(Ctrl* ctrl, const PeerArgs& peer, int lane,
                                                           long long (&got)[kPeerCounters], unsigned long long& epoch_out) {
  const unsigned long long epoch = static_cast<unsigned long long>(ctrl->peer_epoch) + 1ull;
  const int par = static_cast<int>(epoch & 1ull);
  const long long* mine = reinterpret_cast<const long long*>(&ctrl->stats);
#pragma unroll
  for (int k = 0; k < kPeerCounters; ++k) got[k] = 0;
  bool timed_out = false;
  if (lane < peer.world) {
    PeerSlot* dst = peer.buf[lane] + par * kMaxPeers + peer.rank;
#pragma unroll
    for (int k = 0; k < kPeerCounters; ++k) {
      asm volatile("st.relaxed.sys.global.s64 [%0], %1;" ::"l"(&dst->counters[k]), "l"(mine[k]) : "memory");
    }
    st_release_sys_u64(&dst->flag, epoch);  // release: counters (and a grid record stored before) are visible before the flag
    const PeerSlot* src = peer.buf[peer.rank] + par * kMaxPeers + lane;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys_u64(&src->flag) != epoch) {
      if (peer.timeout_ns != 0ull && global_timer_ns() - t0 > peer.timeout_ns) {
        timed_out = true;
        break;
      }
      __nanosleep(100);
    }
    if (!timed_out) {
#pragma unroll
      for (int k = 0; k < kPeerCounters; ++k) {
        asm volatile("ld.relaxed.sys.global.s64 %0, [%1];" : "=l"(got[k]) : "l"(&src->counters[k]) : "memory");
      }
    }
  }
  const unsigned n_to = __popc(__ballot_sync(0xffffffffu, timed_out));
#pragma unroll
  for (int k = 0; k < kPeerCounters; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) got[k] += __shfl_xor_sync(0xffffffffu, got[k], o);
  }
  epoch_out = epoch;
  return n_to;
}

// Publishes the summed counters as ctrl->gx.stats (lane 0 of the exchanging warp).  A peer that did not deliver in time:
// a sum over some of the shards is never published -- the step closes on the shard's own record, and the error is
// STICKY: ctrl->peer_error on the device, the mapped host word for the API, which refuses every further step with
// AS_ERR_PEER (the shards may have promoted differently).
__device__ __forceinline__ void peer_publish(Ctrl* ctrl, const PeerArgs& peer, const long long (&got)[kPeerCounters],
                                             unsigned n_to, unsigned long long epoch) {
  AsStats g = ctrl->stats;  // level, step counter, reward sum: this shard's
  if (n_to == 0) {
    long long* gs = reinterpret_cast<long long*>(&g);
#pragma unroll
    for (int k = 0; k < kPeerCounters; ++k) gs[k] = got[k];
  } else {
    ctrl->peer_timeouts += n_to;
    ctrl->peer_error = 1u;
    if (peer.host_error) {
      *reinterpret_cast<volatile uint32_t*>(peer.host_error) = static_cast<uint32_t>(epoch) | 0x80000000u;
      __threadfence_system();
    }
  }
  ctrl->gx.stats = g;
  ctrl->peer_epoch = static_cast<uint32_t>(epoch == 0xFFFFFFFFull ? 0ull : epoch);
}

// Closes a fused step (one thread, after the fold): decides the promotion of ENV:471 for the next step on `promote_on`
// (this shard's statistics, or their sum over the shards), reports the step's reset count, flips the state parity,
// advances the Philox step counter and empties the reset and regeneration lists for the next step.
__device__ __forceinline__ void close_step(const StepArgs& a, Ctrl* ctrl, const AsStats& promote_on, unsigned n_reset) {
  ctrl->stats_folded = 0;
  ctrl->promote_cur = promotion_decision(a.P, promote_on);
  if (a.rows.n_reset) *a.rows.n_reset = static_cast<int32_t>(a.want_reset_list ? ctrl->n_reset_list : n_reset);
  ctrl->parity ^= 1u;
  ctrl->step_counter += 1ull;
  ctrl->n_reset_list = 0;
  ctrl->n_regen_list = 0;
}

// The last CTA of a fused step kernel (every CTA takes a ticket once its counters are out).  When the launch is
// allowed to close its own step (StepArgs::self_finish: no regeneration kernels behind it, no all-reduce announced) and
// at least one env reset -- so that pass 2 for everybody was the right assumption (DRL:360) -- it folds the statistics
// and closes the step; k_fixup_finish then finds step_state == 2 and returns at once.  Without peers the reset count is
// read before anything is folded: a step in which nobody reset leaves its counters in the slots for k_fixup_finish.
// (The two branches stay apart: merged into one, they change the register allocation of the fused instantiations, and
// the launch-bound small batches, whose step ends with this CTA, measured slower.)
__device__ __forceinline__ void close_step_by_last_cta(const StepArgs& a, Ctrl* ctrl, int lane) {
  __threadfence();
  unsigned state = 1u;
  if (a.self_finish) {
    if (a.peer.world > 0) {
      // sharded, promotion on the global mean: fold, exchange the ten counters with every peer over NVLink (this warp;
      // a peer's last CTA answers when ITS step kernel gets there), then decide on the sums -- the exchange and the
      // finish ride in the step kernel's last CTA instead of two more launches
      const unsigned nr = fold_stats_warp(ctrl, a.num_envs, lane);
      __syncwarp();
      __threadfence();
      long long got[kPeerCounters];
      unsigned long long ep;
      const unsigned n_to = peer_sum_counters_warp(ctrl, a.peer, lane, got, ep);
      if (lane == 0) {
        peer_publish(ctrl, a.peer, got, n_to, ep);
        ctrl->stats_folded = 1;
      }
      __syncwarp();
      const long long global_resets = __shfl_sync(0xffffffffu, n_to == 0 ? got[1] /* AsStats::n_reset */ : static_cast<long long>(nr), 0);
      if (global_resets > 0 || (a.P.flags & AS_FLAG_SKIP_PASS2)) {
        if (lane == 0) close_step(a, ctrl, ctrl->gx.stats, nr);
        state = 2u;
      }  // else: nobody reset anywhere -- k_fixup_finish redoes the step without pass 2, on ctrl->gx (already folded)
    } else if (slot_sum(ctrl, kCntReset) > 0 || (a.P.flags & AS_FLAG_SKIP_PASS2)) {
      const unsigned nr = fold_stats_warp(ctrl, a.num_envs, lane);
      __syncwarp();
      if (lane == 0) close_step(a, ctrl, ctrl->stats, nr);
      state = 2u;
    }
  }
  if (lane == 0) {
    ctrl->blocks_done = 0;
    ctrl->step_state = state;
  }
}

// 3-call path: the last CTA of pass 1 folds its statistics (what k_fold_pass1 did as a launch of its own): consumes the
// promotion every CTA applied, advances the Philox step counter -- a reset that follows draws at the advanced counter.
__device__ __forceinline__ void close_pass1_by_last_cta(const StepArgs& a, Ctrl* ctrl, int lane) {
  __threadfence();
  fold_stats_warp(ctrl, a.num_envs, lane);
  __syncwarp();
  if (lane == 0) {
    ctrl->promote_cur = 0;
    ctrl->step_counter += 1ull;
    ctrl->blocks_done = 0;
  }
}

// ------------------------------------------------------------------------------------------------ the tile
// A CTA is 8 warps on one 128-env tile, two threads per env:
//   warps 0-3  "MDP role"    thread t owns env t: state word, stone window, contact gathers, pass 1, dones, reward,
//                            masked reset, pass 2, head/tail of the observation row
//   warps 4-7  "joint role"  thread t owns env t's three 21-float rows: scaled joint positions, clipped joint
//                            velocities, the reward's energy / action / at-limit sums, and (as a warp) the start
//                            pose of the envs that reset
// The two roles wait on separate mbarriers (root/body tiles vs joint/action tiles), run concurrently, meet at one
// CTA barrier (inputs consumed; sums and reset flags exchanged through shared memory) and then fill disjoint
// columns of the observation tile.  Twice the resident warps of a one-thread-per-env CTA for the same shared
// memory, and half the serial instruction stream per env.
#ifdef AS_TIMING
#define AS_T(var) const long long var = clock64()
#define AS_TACC(slot, from, to) atomicAdd(&ctrl->dbg_t[slot], static_cast<unsigned long long>((to) - (from)))
#else
#define AS_T(var)
#define AS_TACC(slot, from, to)
#endif

// FULL: the tile has all kTile envs (every tile but a ragged last one).  A template parameter because the
// `active` guards it removes are not free: each one ends a basic block, and the step is bound by how well the
// instruction streams of its two roles schedule, not by DRAM (DESIGN.md section 6).
// FAST: the launch uses none of the options -- w,x,y,z quaternions, no per-term reward output, no observation clamp,
// no final observations, courses of the default AS_NUM_STONES stones.  The host checks that (select_step in as_api.cu)
// and the instantiation drops their uniform branches and takes the course length as a constant.
// (Measured: 179.3 -> 176.7 us per 1M-env step.  Also making the per-array "dense" bits compile-time constants
// removes 45 more instructions per warp but ptxas then spills 56 instead of 20 bytes in the MDP role: 184 us.)
// PRE: the launch follows k_prepare* (large batches, two-FMA quotients, contact matrices in device memory): the
// "foot presses" bits of the current stone AND of the stone after it come as one coalesced one-byte record, the stone
// window is known to be valid and is never written here (k_prepare* of the next step refreshes the records whose tag
// went stale) -- no scattered access is left in the hot kernel but the stones 0..2 of an env that resets.
template <int MODE, bool FULL, int EXACT, bool FAST = false, bool PACKED = false, bool PRE = false>
__device__ __forceinline__ void process_tile(const StepArgs& a, int tile, uint32_t& phase_root,
                                             uint32_t& phase_joint, unsigned char* smem) {
  const AsParams& P = a.P;
  const JointConsts& JC = a.jc;
  const bool exact = use_exact_div<EXACT>(JC);
  const int S = FAST ? kS : static_cast<int>(P.num_steps);  // stones per course
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const bool joint_role = warp >= kTile / 32;
  const int t = tid & (kTile - 1);  // env row inside the tile (both roles)
  const int64_t env0 = static_cast<int64_t>(tile) * kTile;
  const int64_t rem = a.num_envs - env0;
  const int n_valid = FULL ? kTile : (rem < kTile ? static_cast<int>(rem) : kTile);
  const bool active = FULL ? true : t < n_valid;
  const int64_t e = env0 + t;

  float* s_jp = reinterpret_cast<float*>(smem + kOffJp);
  float* s_jv = reinterpret_cast<float*>(smem + kOffJv);
  float* s_act = reinterpret_cast<float*>(smem + kOffAct);
  float* s_rp = reinterpret_cast<float*>(smem + kOffRp);
  float* s_rq = reinterpret_cast<float*>(smem + kOffRq);
  float* s_rv = reinterpret_cast<float*>(smem + kOffRv);
  float* s_body = reinterpret_cast<float*>(smem + (PACKED ? kOffBodyPacked : kOffBody));
  const float* s_root = s_rp;  // PACKED: (kTile, 13) rows of root_state_w
  float* s_org = reinterpret_cast<float*>(smem + (PACKED ? kOffOrgPacked : kOffOrg));
  float* s_obs = reinterpret_cast<float*>(smem);
  Misc* misc = reinterpret_cast<Misc*>(smem + kOffMisc);
  const uint32_t bar_root = smem_u32(&misc->mbar_root);
  const uint32_t bar_joint = smem_u32(&misc->mbar_joint);
  Ctrl* ctrl = a.ws.ctrl;

  AS_T(t_start);
  constexpr bool kNeedActions = MODE != kModePass2;
  constexpr bool kPingPong = MODE == kModeFused || MODE == kModeFixup;
  constexpr bool kStats = MODE == kModeFused || MODE == kModePass1;
  // 3-call path, pass 1: like the fused step the kernel ASSUMES that some env resets and runs pass 2 (ENV:567) for
  // the envs that do not -- into the OTHER state buffer and into the observation tile -- while the state and the
  // observation tail as pass 1 leaves them go to the current state buffer and to ws.tail1.  as_step_pass2 then only
  // has to flip the buffers and redo the envs that did reset; as_step_no_reset puts the tails back.
  constexpr bool kSpec = MODE == kModePass1;

  // ---------------------------------------------------------------- HBM -> SMEM (TMA bulk where the view allows)
  const uint32_t dense = a.dense16;
  const uint32_t bm = bulk_mask(dense, n_valid);
  const bool b_jp = bm & kDenseJp;
  const bool b_jv = bm & kDenseJv;
  const bool b_act = kNeedActions && (bm & kDenseAct);
  const bool b_rp = PACKED || (bm & kDenseRp);  // (PACKED: the three arrive together, see below)
  const bool b_rq = PACKED || (bm & kDenseRq);
  const bool b_rv = PACKED || (bm & kDenseRv);
  const bool b_body = bm & kDenseBody;
  const bool b_org = MODE == kModeFused && (bm & kDenseOrg);
  const bool bulk_root = b_rp || b_rq || b_rv || b_body || b_org;
  const bool bulk_joint = b_jp || b_jv || b_act;
  const bool any_coop = !b_jp || !b_jv || (kNeedActions && !b_act) || !b_rp || !b_rq || !b_rv || !b_body ||
                        (MODE == kModeFused && !b_org);
  if (tid == 0) {
    const uint32_t nv = static_cast<uint32_t>(n_valid);
    if (bulk_root) {
      const uint32_t root_bytes = PACKED ? nv * kRootRow * 4
                                         : (b_rp ? nv * 12 : 0) + (b_rq ? nv * 16 : 0) + (b_rv ? nv * 12 : 0);
      mbar_arrive_expect_tx(bar_root, root_bytes + (b_body ? nv * 36 : 0) + (b_org ? nv * 12 : 0));
      if (b_org) bulk_g2s(smem_u32(s_org), a.in.env_origins + env0 * 3, nv * 12, bar_root);
      if (PACKED) {  // root_pos points at column 0 of the (N,13) rows: one copy brings pos, quat, lin vel (and ang vel)
        bulk_g2s(smem_u32(s_rp), a.in.root_pos + env0 * kRootRow, nv * kRootRow * 4, bar_root);
      } else {
        if (b_rp) bulk_g2s(smem_u32(s_rp), a.in.root_pos + env0 * 3, nv * 12, bar_root);
        if (b_rq) bulk_g2s(smem_u32(s_rq), a.in.root_quat + env0 * 4, nv * 16, bar_root);
        if (b_rv) bulk_g2s(smem_u32(s_rv), a.in.root_lin_vel + env0 * 3, nv * 12, bar_root);
      }
      if (b_body && !a.body_from_prepare) bulk_g2s(smem_u32(s_body), a.in.body_pos + env0 * 9, nv * 36, bar_root);
    }
    if (bulk_joint) {
      mbar_arrive_expect_tx(bar_joint, (b_jp ? nv * kJ * 4 : 0) + (b_jv ? nv * kJ * 4 : 0) + (b_act ? nv * kJ * 4 : 0));
      if (b_jp) bulk_g2s(smem_u32(s_jp), a.in.joint_pos + env0 * kJ, nv * kJ * 4, bar_joint);
      if (b_jv) bulk_g2s(smem_u32(s_jv), a.in.joint_vel + env0 * kJ, nv * kJ * 4, bar_joint);
      if (b_act) bulk_g2s(smem_u32(s_act), a.actions + env0 * kJ, nv * kJ * 4, bar_joint);
    }
    if (b_body && a.body_from_prepare) {
      // the dense body rows are being written by k_prepare*, whose last wave this kernel may overlap (programmatic
      // dependent launch): everything else is in flight, this one copy waits for the primary to complete
      if (a.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
      bulk_g2s(smem_u32(s_body), a.in.body_pos + env0 * 9, nv * 36, bar_root);
    }
  }

  // ---------------------------------------------------------------- MDP role: state word + dependent gathers
  const uint32_t parity = ctrl->parity;
  const uint2* st_in = a.ws.state[parity];
  uint2* st_out = (kPingPong || kSpec) ? a.ws.state[parity ^ 1u] : a.ws.state[parity];
  const float4* stones = a.ws.stones + e * S;
  auto stone_at = [&](int i) -> float4 { return ldg64_f4(stones + i); };
  float4* wrow = a.ws.window + e * 4;
  const bool contact_aligned = ((reinterpret_cast<uintptr_t>(a.in.contact_right) | reinterpret_cast<uintptr_t>(
                                    a.in.contact_left)) & 15u) == 0 &&
                               ((a.in.contact_right_stride | a.in.contact_left_stride) & 3) == 0;

  Mdp m{1, 0, 0, 0.0f};
  int level = 0, ep = 0;
  float4 s_prev = make_float4(0, 0, 0, 0), s_curr = s_prev, s_next = s_prev;
  bool win_valid = false, win_dirty = false, w3_pending = false;
  float4* s_w3 = reinterpret_cast<float4*>(smem + kOffW3);
  bool f_r = false, f_l = false, f_r_next = false, f_l_next = false;  // ENV:425 for the current / the following stone
  const float* cr_row = nullptr;
  const float* cl_row = nullptr;
  if (!joint_role && active) {
    const uint2 sw = st_in[e];
    // k_prepare* -- whose last wave this kernel may overlap as its programmatic dependent -- refreshes stale window
    // records and writes the contact norms: both are read only once it has completed
    if (a.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
    // (entry 3, the stone that enters when the window slides, is fetched only by the few envs that do slide)
    const float4 w0 = wrow[0], w1 = wrow[1], w2 = wrow[2];
    m.idx = state_idx(sw.x);
    m.leg = state_leg(sw.x);
    m.count = state_count(sw.x);
    level = state_level(sw.x);
    ep = state_ep(sw.x);
    m.pot = __uint_as_float(sw.y);
    if (MODE != kModePass2) level = min(level + static_cast<int>(ctrl->promote_cur), P.max_level);
    if (kPingPong) ep = min(ep + 1, kMaxEpisodeLength);  // DRL:351
    if (MODE == kModePass1) {
      ep = a.ext_episode_length ? static_cast<int>(min(a.ext_episode_length[e], (int64_t)kMaxEpisodeLength))
                                : min(ep + 1, kMaxEpisodeLength);
    }
    cr_row = a.in.contact_right + e * a.in.contact_right_stride;
    cl_row = a.in.contact_left + e * a.in.contact_left_stride;
    if (PRE || a.use_pre) {  // "foot presses on the current (the following) stone", evaluated by k_prepare* just before
      const unsigned pre = a.ws.contact_pre[e];
      f_r = pre & 1u;
      f_l = pre & 2u;
      f_r_next = pre & 4u;
      f_l_next = pre & 8u;
    } else {  // small batches are launch-bound: the gathers stay in this kernel and a launch is saved
      f_r = contact_norm(cr_row, m.idx, contact_aligned) > P.contact_epsilon;
      f_l = contact_norm(cl_row, m.idx, contact_aligned) > P.contact_epsilon;
    }
    win_valid = PRE || __float_as_int(w0.w) == m.idx;
    if (win_valid) {
      s_prev = w0; s_curr = w1; s_next = w2;
    } else {  // stale cache (first use, or the fix-up re-reading an env the step already advanced): gather
      s_prev = stone_at(window_slot_stone(m.idx, 0, S));
      s_curr = stone_at(window_slot_stone(m.idx, 1, S));
      s_next = stone_at(window_slot_stone(m.idx, 2, S));
    }
  }
  // the index advanced by one: slide the window (the stone entering at the far end is fetched when written back)
  auto slide_window = [&]() {
    s_prev = s_curr;
    s_curr = s_next;
    // The stone that enters is entry 3 of the window record.  Its 32-byte sector came in with entry 2 above, so this
    // load is answered by L1/L2; gathering it from the stone row instead is a DRAM miss in the middle of the MDP
    // role's critical path (almost every warp has a lane that slides).  A second slide in one step (possible only
    // with stop_frames == 1) or a stale record falls back to the gather.
    s_next = (win_valid && !win_dirty) ? wrow[3] : stone_at(min(m.idx + 1, S - 1));
    win_dirty = true;
  };

  // views the bulk path cannot take (strided (N,13) root_state_w slices, full (N,B,3/13) body tensor, ragged tail)
  if (any_coop) {
    if (!b_jp) coop_load<kJ>(s_jp, a.in.joint_pos, a.in.joint_pos_stride, env0, n_valid);
    if (!b_jv) coop_load<kJ>(s_jv, a.in.joint_vel, a.in.joint_vel_stride, env0, n_valid);
    if (kNeedActions && !b_act) coop_load<kJ>(s_act, a.actions, a.actions_stride, env0, n_valid);
    if (!b_rp) coop_load<3>(s_rp, a.in.root_pos, a.in.root_pos_stride, env0, n_valid);
    if (!b_rq) coop_load<4>(s_rq, a.in.root_quat, a.in.root_quat_stride, env0, n_valid);
    if (!b_rv) coop_load<3>(s_rv, a.in.root_lin_vel, a.in.root_lin_vel_stride, env0, n_valid);
    if (MODE == kModeFused && !b_org) coop_load<3>(s_org, a.in.env_origins, 3, env0, n_valid);
    if (!b_body) {
      for (int i = tid; i < n_valid * 9; i += kThreads) {
        const int r = i / 9;
        const int c = i - r * 9;
        const int b = c / 3;
        const int k = c - b * 3;
        const int row = b == 0 ? a.in.right_foot_row : (b == 1 ? a.in.left_foot_row : a.in.torso_row);
        // (12 bytes out of a 52-byte body row, three rows out of an 884-byte env record: L2 fills of 64 bytes, not 128)
        s_body[i] = ldg64_f(a.in.body_pos + (env0 + r) * a.in.body_env_stride + row * a.in.body_row_stride + k);
      }
    }
    __syncthreads();
  }

  // values that cross the CTA barrier in registers
  float h = 0.0f, roll = 0.0f, pitch = 0.0f;
  Vec3 vb{0, 0, 0};
  PassOut po{};
  bool terminated = false, time_out = false, is_reset = false, mirror = false, regen = false;
  bool fell = false, so_fast = false, died = false, missed = false, adv1 = false, adv2 = false;
  float r_partial = 0.0f, r_speed = 0.0f, r_step = 0.0f, r_bonus = 0.0f;
  int idx_after_pass1 = 0;
  const unsigned long long step_now = ctrl->step_counter;
  float o_jp[kJ], o_jv[kJ];
#ifdef AS_TIMING
  long long t_b1a = 0, t_b1b = 0;
#endif

  if (!joint_role) {
    // ================================================================ MDP role, before the barrier
    AS_T(t_m0);  // state word + window + contact norms are in registers (their consumers ran above)
    if (bulk_root) mbar_wait(bar_root, phase_root);
    AS_T(t_m1);
    Vec3 p{0, 0, 0}, v{0, 0, 0}, rf{0, 0, 0}, lf{0, 0, 0};
    float torso_z = 0.0f;
    if (active) {
      if (PACKED) {  // row stride 13 (odd): conflict-free
        p = Vec3{s_root[t * kRootRow], s_root[t * kRootRow + 1], s_root[t * kRootRow + 2]};
        v = Vec3{s_root[t * kRootRow + 7], s_root[t * kRootRow + 8], s_root[t * kRootRow + 9]};
      } else {
        p = Vec3{s_rp[t * 3], s_rp[t * 3 + 1], s_rp[t * 3 + 2]};
        v = Vec3{s_rv[t * 3], s_rv[t * 3 + 1], s_rv[t * 3 + 2]};
      }
      rf = Vec3{s_body[t * 9 + 0], s_body[t * 9 + 1], s_body[t * 9 + 2]};
      lf = Vec3{s_body[t * 9 + 3], s_body[t * 9 + 4], s_body[t * 9 + 5]};
      torso_z = s_body[t * 9 + 8];
    }
    FootGeom geom{};
    Quat inv{1, 0, 0, 0};
    const int idx_before = m.idx;
    float speed = 0.0f;
    if (active && MODE != kModePass2) {
      // ---- dones first, ENV:396-405: they need only the staged root / body rows, and knowing early which envs
      // reset lets their extra loads fly while pass 1 is being computed
      h = torso_z - min_nan(lf.z, rf.z);  // ENV:281-283
      time_out = ep >= P.max_episode_length - 1;
      fell = h < P.termination_height[level];
      speed = norm3(v.x, v.y, v.z);
      so_fast = speed > P.max_root_speed;
      died = p.z < P.termination_height_absolute;
      if (P.flags & AS_FLAG_MISSED_STEP) {
        // extension: the swing foot is down (below the stone it heads for) outside that stone's footprint; leg and
        // stone as they are before this pass updates them
        const float dsw = m.leg ? norm2(lf.x - s_curr.x, lf.y - s_curr.y) : norm2(rf.x - s_curr.x, rf.y - s_curr.y);
        missed = ((m.leg ? lf.z : rf.z) < s_curr.z + P.missed_step_height) && dsw >= P.step_radius;
      }
      terminated = fell || so_fast || died || missed;
      is_reset = terminated || time_out;
      // an env that resets restarts on stones 0..3 (one 64-byte record at the head of its stone row): start
      // pulling it in now, it is read after pass 1
      if (MODE == kModeFused && is_reset) {
        prefetch_l1(stones);
      }
    }
    unsigned rmask = 0, rbase = 0;
    if (MODE == kModeFused) {  // the joint role finishes the envs that reset: tell it early which ones they are
      misc->flags[t] = is_reset ? 1u : 0u;
      flags_arrive();
    }
    if (MODE == kModeFused || kSpec) {
      // reserve this warp's range of the reset-id list now: the atomic's round trip to L2 (the ids are written at
      // the end) then hides behind pass 1 instead of sitting in front of the hand-off to the joint role
      // (3-call path: the list lets as_reset take "the envs pass 1 flagged" without a host round trip)
      rmask = __ballot_sync(0xffffffffu, is_reset);
      if (rmask && (kSpec || a.want_reset_list) && lane == __ffs(rmask) - 1)
        rbase = atomicAdd(&ctrl->n_reset_list, __popc(rmask));
    }
    bool moved1 = false;
    if (active) {
      h = torso_z - min_nan(lf.z, rf.z);   // ENV:281-283
      geom = foot_geometry(P, rf, lf, f_r, f_l, s_curr);
      moved1 = foot_update(P, geom, m, po, S);
      if (moved1) slide_window();
    }
    orient_wait();  // roll / pitch / quat_inv of this env were computed by the joint role (ENV:285, MATH:238-248)
    if (active) {
      inv = Quat{misc->x_inv[0][t], misc->x_inv[1][t], misc->x_inv[2][t], misc->x_inv[3][t]};
      targets_and_potential(P, a.inv_step_dt, exact, p, inv, s_prev, s_curr, s_next, m, po);
      adv1 = po.advanced;
      idx_after_pass1 = m.idx;
      if (MODE != kModePass2) {
        // ---- reward terms that do not need the joint sums, ENV:350-375
        const float r_progress = m.pot - po.old_pot;
        r_speed = speed > 1.6f ? speed - 1.6f : 0.0f;
        r_partial = P.alive_reward_scale + r_progress;  // head of the reference's left-to-right sum, ENV:378-380
        if (!FAST && a.out.reward_terms) {
          float* rt = a.out.reward_terms + e * AS_NUM_REWARD_TERMS;
          rt[0] = P.alive_reward_scale; rt[1] = r_progress; rt[4] = r_speed;
        }
        const bool pays_step = po.reached && m.count == 1 && m.idx < S - 1;
        r_step = pays_step ? 50.0f * expf((-po.d_swing) / 0.25f) : 0.0f;
        r_bonus = (m.idx == S - 1 && po.body_dist < 0.15f) ? 10.0f : 0.0f;
      }
    }

    if (kSpec && active) {
      uint2 v1;
      v1.x = pack_state(m.idx, m.leg, m.count, level, ep);
      v1.y = __float_as_uint(m.pot);
      a.ws.state[parity][e] = v1;
      float4* t1 = a.ws.tail1 + e * 3;
      t1[0] = make_float4(po.contact_r, po.contact_l, po.tb0.x, po.tb0.y);
      t1[1] = make_float4(po.tb0.z, po.tb1.x, po.tb1.y, po.tb1.z);
      t1[2] = make_float4(po.tb2.x, po.tb2.y, po.tb2.z, 0.0f);
      a.ws.pass1_reset[e] = is_reset ? 1 : 0;
    }
    if ((MODE == kModeFused || kSpec) && active) {
      if (MODE == kModeFused && is_reset) {
        if (!FAST && a.out.final_obs) {
          // final observation (AsStepOut.final_obs): head and tail of the row as pass 1 left them, before the reset
          // below overwrites them; roll / pitch / v_b follow once the joint role has published them
          float* fin = a.out.final_obs + e * kObs;
          const float c = a.out.obs_clip;
          fin[0] = clip_obs(h, c);
          fin[48] = clip_obs(po.contact_r, c); fin[49] = clip_obs(po.contact_l, c);
          fin[50] = clip_obs(po.tb0.x, c); fin[51] = clip_obs(po.tb0.y, c); fin[52] = clip_obs(po.tb0.z, c);
          fin[53] = clip_obs(po.tb1.x, c); fin[54] = clip_obs(po.tb1.y, c); fin[55] = clip_obs(po.tb1.z, c);
          fin[56] = clip_obs(po.tb2.x, c); fin[57] = clip_obs(po.tb2.y, c); fin[58] = clip_obs(po.tb2.z, c);
        }
        mirror = misc->coin[t] != 0;  // drawn by the joint role in its idle time (ordered by the orientation barrier)
        // ---- masked reset, ENV:487-538.  Pass 2 on the post-reset state: identity orientation (vector part +-0),
        // zero velocity, zero contacts (contact_sensor.py:155), stale body positions; so roll = pitch = v_b = 0 and
        // targets_b = stone - root.  The start-pose joints are produced by the joint-role warps.
        regen = ((P.flags & AS_FLAG_INTENDED_REGEN) && m.idx > S / 2) || (P.flags & AS_FLAG_GRID_CURRICULUM);
        const Vec3 org{s_org[t * 3], s_org[t * 3 + 1], s_org[t * 3 + 2]};
        p = Vec3{P.default_root_pos[0] + org.x, P.default_root_pos[1] + org.y, P.default_root_pos[2] + org.z};
        if (regen) {
          first_three_stones(P, org, s_prev, s_curr, s_next);
        } else {
          s_prev = stone_at(0);
          s_curr = stone_at(1);
          s_next = stone_at(2);
        }
        win_dirty = true;
        m.count = 0;
        m.leg = mirror ? 1 : 0;  // ENV:491,538
        m.idx = 1;
        ep = 0;  // DRL:584
        po.contact_r = 0.0f;
        po.contact_l = 0.0f;
        po.tb0 = Vec3{s_prev.x - p.x, s_prev.y - p.y, s_prev.z - p.z};
        po.tb1 = Vec3{s_curr.x - p.x, s_curr.y - p.y, s_curr.z - p.z};
        po.tb2 = Vec3{s_next.x - p.x, s_next.y - p.y, s_next.z - p.z};
        po.body_dist = norm2(s_next.x - p.x, s_next.y - p.y);
        m.pot = potential_of(P, a.inv_step_dt, po.body_dist, exact);  // ENV:487-488, then ENV:415-416 in pass 2
      } else if (!(P.flags & AS_FLAG_SKIP_PASS2) && !(kSpec && is_reset)) {
        // ---- pass 2 over ALL envs, ENV:567 (SURVEY D7), on unchanged physics: only the foot state machine can
        // change anything.  Assumed to happen; the fix-up kernel undoes the assumption when no env reset.
        if (idx_after_pass1 != idx_before) {  // the current stone changed in pass 1: new contact column
          if (PRE) {  // (the index moved by exactly one: the record's second pair)
            f_r = f_r_next;
            f_l = f_l_next;
          } else {
            f_r = contact_norm(cr_row, m.idx, contact_aligned) > P.contact_epsilon;
            f_l = contact_norm(cl_row, m.idx, contact_aligned) > P.contact_epsilon;
          }
          geom = foot_geometry(P, rf, lf, f_r, f_l, s_curr);
        }
        const bool moved = foot_update(P, geom, m, po, S);
        adv2 = po.advanced;  // (taken back with pass 2 by k_fixup_finish, k_pass2_revert or k_pass2_commit)
        if (moved) {
          slide_window();
          targets_and_potential(P, a.inv_step_dt, exact, p, inv, s_prev, s_curr, s_next, m, po);
        }
        // (unmoved: targets, body distance and potential are recomputed to the same values; old_potentials is dead)
      }
    }
    if (active) {
      uint2 sw;
      sw.x = pack_state(m.idx, m.leg, m.count, level, ep);
      sw.y = __float_as_uint(m.pot);
      if (PRE) st_keep_u2(st_out + e, sw, policy_evict_last());  // (k_prepare* of the next step reads it first thing)
      else st_out[e] = sw;
      if (PRE) {
        // this instantiation never writes windows: tell k_prepare* of the next step which records to refresh
        const unsigned stale = __ballot_sync(0xffffffffu, win_dirty);
        if (lane == 0) a.ws.win_stale[e >> 5] = stale;
      }
      if (!PRE && (win_dirty || !win_valid) && !regen) {  // (a regenerated env's window is written by the regeneration kernel)
        s_prev.w = __int_as_float(m.idx);  // tag
        wrow[0] = s_prev; wrow[1] = s_curr; wrow[2] = s_next;
        // Entry 3 is a stone this step never looked at: a gather out of the stone row.  Loading it into a register
        // and storing it would park the warp on the store until DRAM answers (in-order issue), in the middle of the
        // MDP role's critical path and for nearly every warp; instead it travels global -> shared asynchronously
        // and is written back at the very end of the tile.
        cp_async16(smem_u32(s_w3 + t), stones + window_slot_stone(m.idx, 3, S));
        w3_pending = true;
      }
    }
#ifdef AS_TIMING
    if (tid == 0) { AS_T(t_m2); AS_TACC(0, t_start, t_m0); AS_TACC(1, t_m0, t_m1); AS_TACC(2, t_m1, t_m2); }
#endif
    if (kSpec && rmask) {
      const unsigned base = __shfl_sync(0xffffffffu, rbase, __ffs(rmask) - 1);
      if (is_reset) a.ws.reset_ids[base + __popc(rmask & ((1u << lane) - 1u))] = static_cast<int32_t>(e);
    }
    if (MODE == kModeFused) {
      // ---- reset / regeneration id lists (warp ballots)
      if (rmask && a.want_reset_list) {
        const unsigned base = __shfl_sync(0xffffffffu, rbase, __ffs(rmask) - 1);
        int32_t* ids_dst = a.rows.reset_ids ? a.rows.reset_ids : a.ws.reset_ids;
        if (is_reset) ids_dst[base + __popc(rmask & ((1u << lane) - 1u))] = static_cast<int32_t>(e);
      }
      const unsigned gmask = __ballot_sync(0xffffffffu, regen);
      if (gmask) {
        const int leader = __ffs(gmask) - 1;
        unsigned base = 0;
        if (lane == leader) base = atomicAdd(&ctrl->n_regen_list, __popc(gmask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (regen) {
          const unsigned pos = base + __popc(gmask & ((1u << lane) - 1u));
          a.ws.regen_ids[pos] = static_cast<int32_t>(e);
          a.ws.regen_info[pos] = static_cast<uint8_t>(idx_after_pass1);  // where the episode ended
        }
      }
    }
  } else {
    // ================================================================ joint role, before the barrier
    // The root tile is small and lands first: do the orientation math of this env (ENV:285,293; MATH:238-248) while
    // the three joint tiles are still in flight, and hand roll / pitch / quat_inv to the MDP role.
    // The mirror coin of every env (ENV:518; draw 0 of the reset stream): ten Philox rounds that the MDP role would
    // otherwise run, in three warps out of four, on its critical path; here they fill the wait for the first tiles.
    bool my_coin = false;
    if (MODE == kModeFused && active) {
      const uint4 rblk = philox_block(P.seed, step_now, kStreamReset, static_cast<uint32_t>(e + a.env_id_offset), 0);
      my_coin = u32_to_unit(rblk.x) > 0.5f;
      misc->coin[t] = my_coin ? 1 : 0;
    }
    if (bulk_root) mbar_wait(bar_root, phase_root);
    Quat q{1, 0, 0, 0};
    if (active) {
      const float4 q4 = PACKED ? make_float4(s_root[t * kRootRow + 3], s_root[t * kRootRow + 4], s_root[t * kRootRow + 5],
                                             s_root[t * kRootRow + 6])
                               : *reinterpret_cast<const float4*>(s_rq + t * 4);
      q = (!FAST && a.in.quat_xyzw) ? Quat{q4.w, q4.x, q4.y, q4.z} : Quat{q4.x, q4.y, q4.z, q4.w};
      const Quat inv = quat_inverse(q);  // first: the MDP role is waiting for it to transform the targets
      misc->x_inv[0][t] = inv.w; misc->x_inv[1][t] = inv.x; misc->x_inv[2][t] = inv.y; misc->x_inv[3][t] = inv.z;
    }
    orient_arrive();  // (warp-convergent: outside the `active` branch)
    if (active) {
      const Vec3 v = PACKED ? Vec3{s_root[t * kRootRow + 7], s_root[t * kRootRow + 8], s_root[t * kRootRow + 9]}
                            : Vec3{s_rv[t * 3], s_rv[t * 3 + 1], s_rv[t * 3 + 2]};
      euler_roll_pitch(q, roll, pitch);  // read by the MDP role only after the sums hand-off further down
      vb = rotate_by_inverse(q, v);
      misc->x_roll[t] = roll;
      misc->x_pitch[t] = pitch;
      misc->x_vb[0][t] = vb.x; misc->x_vb[1][t] = vb.y; misc->x_vb[2][t] = vb.z;
    }
    // (nothing but the loop's own 42 outputs and three sums stays in registers across it: roll / pitch / v_b and the
    // coin are read back from shared memory afterwards -- a spilled value costs more than the round trip)
    if (bulk_joint) mbar_wait(bar_joint, phase_joint);
    AS_T(t_j0);
    float energy = 0.0f, act_sq = 0.0f;
    int at_limit = 0;
    if (active) {
      const float* my_jp = s_jp + t * kJ;
      const float* my_jv = s_jv + t * kJ;
      const float* my_act = s_act + t * kJ;
      auto joint_rows = [&](auto ex) {
#pragma unroll
        for (int j = 0; j < kJ; ++j) {
          const float jv = my_jv[j];
          const float sc = scale_joint(JC.c[j], my_jp[j], decltype(ex)::value);  // ENV:287-291
          if (kNeedActions) {
            const float act = clamp_nan(my_act[j], -1.0f, 1.0f);  // ENV:268
            at_limit += fabsf(sc) > JC.c[j].w ? 1 : 0;               // ENV:367 (0.99; rides in the record's 4th word)
            energy += fabsf(jv * act);                               // ENV:365
            act_sq = fmaf(act, act, act_sq);                         // ENV:364
          }
          o_jp[j] = sc;
          o_jv[j] = clamp_nan(jv * P.dof_vel_scale, -5.0f, 5.0f);  // ENV:337
        }
      };
      // (one copy of the loop per choice: with EXACT == 2 the choice is made here, once, not in every iteration)
      if (exact) joint_rows(std::true_type{});
      else joint_rows(std::false_type{});
    }
#ifdef AS_TIMING
    if (tid == kTile) { AS_T(t_j1); AS_TACC(8, t_start, t_j0); AS_TACC(9, t_j0, t_j1); }
#endif
    if (kNeedActions) {
      misc->red_energy[t] = energy;
      misc->red_actsq[t] = act_sq;
      misc->red_limit[t] = at_limit;
    }
    // The joint role does not wait for the MDP role: once all FOUR joint warps have consumed their rows the
    // observation tile may be written; the MDP role is told the same (and that the sums are ready), and it told us
    // earlier which envs reset.
#ifdef AS_TIMING
    t_b1a = clock64();
#endif
    joint_rows_consumed();
    sums_arrive();
    if (MODE == kModeFused) flags_wait();
#ifdef AS_TIMING
    t_b1b = clock64();
#endif
    if (active) {
      float* row = s_obs + t * kObs;
      // an env that reset is observed in its start pose: identity orientation, zero velocity (pass 2, ENV:567)
      const bool was_reset = MODE == kModeFused && (misc->flags[t] & 1u);
      row[1] = was_reset ? 0.0f : misc->x_roll[t];
      row[2] = was_reset ? 0.0f : misc->x_pitch[t];
      row[3] = was_reset ? 0.0f : misc->x_vb[0][t];
      row[4] = was_reset ? 0.0f : misc->x_vb[1][t];
      row[5] = was_reset ? 0.0f : misc->x_vb[2][t];
#pragma unroll
      for (int j = 0; j < kJ; ++j) {
        row[6 + j] = o_jp[j];
        row[6 + kJ + j] = o_jv[j];
      }
    }
    if (MODE == kModeFused) {
      // Envs that reset are finished by the whole warp: lane j produces joint j of the start pose (ENV:505-560) and
      // stores it both into the observation row (as joint_pos_scaled, what pass 2 sees) and, coalesced, into the
      // start-pose rows handed to PhysX (ENV:563-565).
      const unsigned fl = misc->flags[t];
      unsigned todo = __ballot_sync(0xffffffffu, (fl & 1u) != 0);
      __syncwarp();
      const int row0 = (warp - kTile / 32) * 32;
      // The joint noise of an env (ENV:542-560) is draws 1..21 of its reset stream: six Philox blocks.  They are drawn
      // for FIVE envs per pass -- lane (slot, block) = (lane / 6, lane % 6) -- and parked in shared memory, where lane j
      // picks up draw 1 + j: a warp with n resets runs ceil(n / 5) passes of ten rounds instead of n.  The warp with
      // the most resets is the one its CTA waits for.
      uint4* phx = reinterpret_cast<uint4*>(smem + kOffPhx) + row0;
      const uint32_t* phx_w = reinterpret_cast<const uint32_t*>(phx);
      auto philox_group = [&](unsigned mask) {  // blocks of the first five set bits of `mask`
        const int slot = lane / 6, blk = lane - slot * 6;
        int my_r = -1;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          if (k == slot && mask) my_r = __ffs(mask) - 1;
          mask &= mask - 1u;
        }
        uint4 b = make_uint4(0u, 0u, 0u, 0u);
        if (my_r >= 0 && lane < 30) {
          const uint32_t gid_g = static_cast<uint32_t>(env0 + row0 + my_r + a.env_id_offset);
          b = philox_block(P.seed, step_now, kStreamReset, gid_g, static_cast<uint32_t>(blk));
        }
        phx[lane] = b;
      };
      int k5 = 5;  // position of the next env in its group of five (5: draw a new group first)
      const ResetTables& T = misc->rt;
      const float4 jc_l = T.jc[lane];
      const float pose_l = T.pose[lane], pose_m_l = T.pose_mirrored[lane], vel_m_l = T.vel_mirrored[lane];
      while (todo) {
        if (k5 == 5) {
          __syncwarp();
          philox_group(todo);
          __syncwarp();
          k5 = 0;
        }
        const int r = __ffs(todo) - 1;
        todo &= todo - 1u;
        const bool mirror_r = misc->coin[row0 + r] != 0;
        const int64_t e_r = env0 + row0 + r;
        if (lane < kJ) {
          const int d = 1 + lane;  // draw d = component d % 4 of block d / 4
          const float u = u32_to_unit(phx_w[(k5 * 6 + (d >> 2)) * 4 + (d & 3)]);
          const float val = reset_joint_value(P, mirror_r ? pose_m_l : pose_l, jc_l, u, exact);
          float* row = s_obs + (row0 + r) * kObs;
          if (!FAST && a.out.final_obs) {  // final observation: the pass-1 joint columns, before the start pose replaces them
            float* fin = a.out.final_obs + e_r * kObs;
            fin[6 + lane] = clip_obs(row[6 + lane], a.out.obs_clip);
            fin[6 + kJ + lane] = clip_obs(row[6 + kJ + lane], a.out.obs_clip);
          }
          row[6 + lane] = scale_joint(jc_l, val, exact);
          const float jv0 = mirror_r ? vel_m_l : 0.0f;
          row[6 + kJ + lane] = clamp_nan(jv0 * P.dof_vel_scale, -5.0f, 5.0f);
          if (a.rows.joint_pos) a.rows.joint_pos[e_r * kJ + lane] = val;
          if (a.rows.joint_vel) a.rows.joint_vel[e_r * kJ + lane] = jv0;
        }
        if (a.rows.root_state && lane < AS_ROOT_STATE_DIM) {
          const float z = mirror_r ? -0.0f : 0.0f;  // ENV:535 flips the sign of the (zero) vector part
          float val = 0.0f;
          if (lane < 3) {
            const float d = lane == 0 ? P.default_root_pos[0] : (lane == 1 ? P.default_root_pos[1] : P.default_root_pos[2]);
            val = d + s_org[(row0 + r) * 3 + lane];  // ENV:515
          } else if (lane == 3) {
            val = 1.0f;
          } else if (lane <= 6) {
            val = z;
          }
          a.rows.root_state[e_r * AS_ROOT_STATE_DIM + lane] = val;
        }
        ++k5;
      }
    }
  }
  if (bulk_root) phase_root ^= 1u;
  if (bulk_joint) phase_joint ^= 1u;

  float reward = 0.0f;
  if (!joint_role) {
    // ================================================================ MDP role, once the joint rows are consumed
#ifdef AS_TIMING
    t_b1a = clock64();
#endif
    sums_wait();
#ifdef AS_TIMING
    t_b1b = clock64();
#endif
    if (MODE != kModePass2 && active) {  // reward, ENV:377-394
      const float r_energy = P.energy_cost_scale * misc->red_energy[t];
      const float r_action = P.actions_cost_scale * sqrt_rn(misc->red_actsq[t]);
      const float r_limit = static_cast<float>(misc->red_limit[t]) * P.joint_at_limit_cost_scale;
      // roll / pitch were written by the joint role before it signalled the sums (ENV:356-359)
      const float roll_j = misc->x_roll[t], pitch_j = misc->x_pitch[t];
      const float r_roll = (roll_j > 0.4f || roll_j < -0.4f) ? fabsf(roll_j) : 0.0f;
      const float r_pitch = (pitch_j > 0.4f || pitch_j < -0.2f) ? fabsf(pitch_j) : 0.0f;
      float total = r_partial - r_roll;
      total = total - r_pitch;
      total = total - r_speed;
      total = total - r_energy;
      total = total - r_action;
      total = total - r_limit;
      total = total + r_step;
      total = total + r_bonus;
      reward = terminated ? P.death_cost : total;
      a.out.reward[e] = reward;
      a.out.terminated[e] = terminated ? 1 : 0;
      a.out.time_out[e] = time_out ? 1 : 0;
      if (a.out.dones) a.out.dones[e] = is_reset ? 1 : 0;
      if (!FAST && a.out.reward_terms) {
        float* rt = a.out.reward_terms + e * AS_NUM_REWARD_TERMS;
        rt[2] = r_roll; rt[3] = r_pitch;
        rt[5] = r_energy; rt[6] = r_action; rt[7] = r_limit; rt[8] = r_step; rt[9] = r_bonus;
      }
      if (MODE == kModeFused && !FAST && a.out.final_obs && is_reset) {  // the rest of the final observation's head
        float* fin = a.out.final_obs + e * kObs;
        const float c = a.out.obs_clip;
        fin[1] = clip_obs(roll_j, c);
        fin[2] = clip_obs(pitch_j, c);
        fin[3] = clip_obs(misc->x_vb[0][t], c);
        fin[4] = clip_obs(misc->x_vb[1][t], c);
        fin[5] = clip_obs(misc->x_vb[2][t], c);
      }
    }
    if (active) {  // head and tail of the observation row, ENV:330-343
      float* row = s_obs + t * kObs;
      row[0] = h;
      row[48] = po.contact_r;
      row[49] = po.contact_l;
      row[50] = po.tb0.x; row[51] = po.tb0.y; row[52] = po.tb0.z;
      row[53] = po.tb1.x; row[54] = po.tb1.y; row[55] = po.tb1.z;
      row[56] = po.tb2.x; row[57] = po.tb2.y; row[58] = po.tb2.z;
    }
    if (kStats) {  // packed warp reductions of the step counters
      const unsigned w0 = (is_reset ? 1u : 0u) | (terminated ? 1u << 8 : 0u) | (time_out ? 1u << 16 : 0u) |
                          (fell ? 1u << 24 : 0u);
      const unsigned w1 = (so_fast ? 1u : 0u) | (died ? 1u << 8 : 0u) | (adv1 ? 1u << 16 : 0u) |
                          (adv2 ? 1u << 24 : 0u);
      const unsigned w2 = (regen ? 1u : 0u) | (static_cast<unsigned>(active ? idx_after_pass1 : 0) << 8) |
                          (missed ? 1u << 20 : 0u);
      const unsigned s0 = __reduce_add_sync(0xffffffffu, w0);
      const unsigned s1 = __reduce_add_sync(0xffffffffu, w1);
      const unsigned s2 = __reduce_add_sync(0xffffffffu, w2);
      const unsigned lmax = __reduce_max_sync(0xffffffffu, static_cast<unsigned>(active ? level : 0));
      float rs = active ? reward : 0.0f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
      if (lane == 0) {
        unsigned* wc = misc->wcnt[warp];
        wc[kCntReset] = s0 & 255u;
        wc[kCntTerminated] = (s0 >> 8) & 255u;
        wc[kCntTimeOut] = (s0 >> 16) & 255u;
        wc[kCntFell] = s0 >> 24;
        wc[kCntSoFast] = s1 & 255u;
        wc[kCntDied] = (s1 >> 8) & 255u;
        wc[kCntAdvanced1] = (s1 >> 16) & 255u;
        wc[kCntAdvanced2] = s1 >> 24;
        wc[kCntRegen] = s2 & 255u;
        wc[kCntSumIndex] = (s2 >> 8) & 4095u;
        wc[kCntMissed] = s2 >> 20;
        wc[kCntLevelMax] = lmax;
        misc->wreward[warp] = rs;
      }
    }
  }

  // ---------------------------------------------------------------- observation tile -> HBM, ENV:326-345
  AS_T(t_post);
  float* obs_dst = a.out.obs + env0 * kObs;
  const bool b_obs = bm & kDenseObs;
  if (!FAST && a.out.obs_clip > 0.0f) {
    // RL-wrapper epilogue (isaaclab_rl/rl_games.py:293): clamp the finished tile in place.  Comparisons, not
    // fminf/fmaxf: torch.clamp hands NaN through.
    const float c = a.out.obs_clip;
    __syncthreads();
    for (int i = tid; i < n_valid * kObs; i += kThreads) {
      const float v = s_obs[i];
      s_obs[i] = v < -c ? -c : (v > c ? c : v);
    }
  }
  if (b_obs) {
    fence_proxy_async_smem();  // make the generic-proxy writes visible to the TMA engine
    __syncthreads();
    if (tid == 0) {
      bulk_s2g(obs_dst, smem_u32(s_obs), static_cast<uint32_t>(n_valid) * kObs * 4);
      bulk_commit();
    }
#ifdef AS_TIMING
    if (tid == 0 || tid == kTile) { AS_T(t_b2); AS_TACC(tid == 0 ? 3 : 10, t_b1a, t_b1b); AS_TACC(tid == 0 ? 4 : 11, t_b1b, t_post); AS_TACC(tid == 0 ? 5 : 12, t_post, t_b2); }
#endif
  } else {
    __syncthreads();
    for (int i = tid; i < n_valid * kObs; i += kThreads) obs_dst[i] = s_obs[i];
  }
  if (kSpec && !FAST && a.out.final_obs && !joint_role) {
    // final observations: pass 1 skipped pass 2 for the envs it flagged, so their finished (clamped) rows of the tile
    // are the rows to keep -- copied by the env's MDP-role warp, one coalesced row at a time
    unsigned todo = __ballot_sync(0xffffffffu, is_reset);
    while (todo) {
      const int r = warp * 32 + __ffs(todo) - 1;
      todo &= todo - 1u;
      const float* src = s_obs + r * kObs;
      float* fin = a.out.final_obs + (env0 + r) * kObs;
      fin[lane] = src[lane];
      if (lane < kObs - 32) fin[32 + lane] = src[32 + lane];
    }
  }
  unsigned ticket = 0;
  if (kStats && warp == 0) {  // CTA totals -> one replicated global slot (fire and forget), by the first warp
    const int slot = blockIdx.x & (kSlots - 1);
    if (lane < kNumCounters) {
      unsigned tot = 0;
#pragma unroll
      for (int w = 0; w < kTile / 32; ++w) tot = lane == kCntLevelMax ? max(tot, misc->wcnt[w][lane]) : tot + misc->wcnt[w][lane];
      if (tot) {
        if (lane == kCntLevelMax) atomicMax(&ctrl->slots[slot][lane], tot);
        else atomicAdd(&ctrl->slots[slot][lane], tot);
      }
    } else if (lane == kNumCounters) {
      float rs = 0.0f;
#pragma unroll
      for (int w = 0; w < kTile / 32; ++w) rs += misc->wreward[w];
      atomicAdd(&ctrl->slot_reward[slot], rs);
    }
    if (MODE == kModeFused || kSpec) {
      // "last CTA closes the step": a ticket per CTA, taken after this CTA's counters are out (fence), by the one
      // thread that has to wait for the bulk store anyway -- the atomic's round trip hides behind that wait
      __syncwarp();
      if (lane == 0) {
        __threadfence();
        ticket = atomicAdd(&ctrl->blocks_done, 1u) + 1u;
      }
    }
  }
#ifdef AS_TIMING
  AS_T(t_w0);
#endif
  if (!PRE && !joint_role) {  // deferred write-back of window entry 3 (the copy was issued microseconds ago)
    cp_async_wait_all();
    if (w3_pending) wrow[3] = s_w3[t];
  }
  if (tid == 0 && b_obs) bulk_wait_read_all();  // shared memory must stay intact until the engine has read it
  if ((MODE == kModeFused || kSpec) && warp == 0) {
    const bool last = __shfl_sync(0xffffffffu, ticket, 0) == static_cast<unsigned>(a.num_tiles);
    if (last) {
      if (kSpec) close_pass1_by_last_cta(a, ctrl, lane);
      else close_step_by_last_cta(a, ctrl, lane);
    }
  }
#ifdef AS_TIMING
  if (tid == 0) { AS_T(t_w1); AS_TACC(6, t_w0, t_w1); AS_TACC(7, t_start, t_w1); atomicAdd(&ctrl->dbg_t[15], 1ull); }
#endif
}

// ------------------------------------------------------------------------------------------------ kernels
// k_prepare*: everything data-dependent and scattered that a step reads, done by a kernel of its own at full occupancy
// with nothing else on its critical path, and handed to the step kernel as coalesced records:
//   * for every env the norms of the 12-byte contact-force vectors of its CURRENT stone and of the stone AFTER it (the
//     one pass 2 looks at when pass 1 advances the index) out of the two (N,1,S,3) PhysX matrices, ENV:421-425 -- the
//     two vectors are neighbours in the row, so the second one rides in the same 64-byte fills as the first;
//   * the stone window of every env whose record went stale (the index moved or the env reset in the last step):
//     stones idx-1 .. idx+2 out of its S x 16-byte stone row, tagged with idx -- the step kernel only reads windows;
//   * optionally the three body rows the task reads (right foot, left foot, torso: 12 bytes each) out of a strided
//     (N,B,13) body_state_w tensor into a dense (N,3,3) array the step kernel takes by bulk copy.
// These random DRAM reads are what floors the step (profiles/r01_membound_probe.txt); issued from inside the step
// kernel they stall a 46-KB CTA each.
struct PrepareArgs {
  AsStateIn in;
  Workspace ws;
  int64_t num_envs;
  float* body_dense;  // non-null: gather the body rows
  int32_t lean;       // the contact matrices live in pinned HOST memory (read across PCIe, where every request counts):
                      // only the current stone's vectors are fetched -- one request per foot and env; the step kernel
                      // instantiation that can gather for itself then fetches the next stone's for the few envs whose
                      // pass 1 advances the index
  int32_t stop_frames;  // ENV:56: pass 1 can advance the index only if the reach counter is one short of this
  float contact_epsilon;  // ENV:425
  int32_t num_stones;     // S, the course length
};

__device__ __forceinline__ void refresh_window_entry(const Workspace& ws, int64_t e, int idx, int slot, int S) {
  float4 v = ldg64_f4(ws.stones + e * S + window_slot_stone(idx, slot, S));
  if (slot == 0) v.w = __int_as_float(idx);  // tag
  ws.window[e * 4 + slot] = v;
}

// One lane per env (rows that are not 16-byte aligned).
__global__ void __launch_bounds__(256) k_prepare(const __grid_constant__ PrepareArgs a) {
  asm volatile("griddepcontrol.launch_dependents;");
  const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= a.num_envs) return;
  const AsStateIn& in = a.in;
  const uint32_t word = a.ws.state[a.ws.ctrl->parity][e].x;
  const int idx = state_idx(word);
  const int nxt = min(idx + 1, a.num_stones - 1);
  const bool stale = (a.ws.win_stale[e >> 5] >> (e & 31)) & 1u;
  const float* rr = in.contact_right + e * in.contact_right_stride;
  const float* lr = in.contact_left + e * in.contact_left_stride;
  // (the next stone's vectors only where pass 1 can advance the index at all: reach counter one short of stop_frames)
  const bool want_next = state_count(word) + 1 >= a.stop_frames;
  const float eps = a.contact_epsilon;
  a.ws.contact_pre[e] = static_cast<uint8_t>(
      (contact_norm(rr, idx, false) > eps ? 1u : 0u) | (contact_norm(lr, idx, false) > eps ? 2u : 0u) |
      ((want_next && contact_norm(rr, nxt, false) > eps) ? 4u : 0u) |
      ((want_next && contact_norm(lr, nxt, false) > eps) ? 8u : 0u));
  if (stale) {
#pragma unroll
    for (int k = 0; k < 4; ++k) refresh_window_entry(a.ws, e, idx, k, a.num_stones);
  }
  if (a.body_dense) {
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const int row = b == 0 ? in.right_foot_row : (b == 1 ? in.left_foot_row : in.torso_row);
      const float* src = in.body_pos + e * in.body_env_stride + row * in.body_row_stride;
#pragma unroll
      for (int k = 0; k < 3; ++k) a.body_dense[e * 9 + b * 3 + k] = ldg64_f(src + k);
    }
  }
}

// TWO lanes per env: the even lane fetches the 16-byte chunk the current stone's vector starts in, the odd lane the
// following chunk, in ONE load instruction per foot -- the two chunks travel as one request whenever they share a
// 128-byte line, which is what counts when the matrices live in pinned host memory: PCIe reads are bound by the number
// of requests in flight, not by their size (tools/e2e_probe.py).  The six floats of the two vectors start at float
// k = (3 idx) & 3 of the first chunk: for k = 3 they run into a third chunk, which the even lane fetches too.
// Needs 16-byte aligned rows.
__global__ void __launch_bounds__(256) k_prepare_paired(const __grid_constant__ PrepareArgs a) {
  asm volatile("griddepcontrol.launch_dependents;");  // the step kernel may stage its tiles under our last wave
  const AsStateIn& in = a.in;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t e = t >> 1;
  const bool live = e < a.num_envs;  // both lanes of a pair agree; no early exit, the shuffles below need the warp
  const int half = static_cast<int>(t & 1);
  const uint32_t word = live ? a.ws.state[a.ws.ctrl->parity][e].x : 0u;
  const int idx = state_idx(word);
  const bool stale = live && ((a.ws.win_stale[e >> 5] >> (e & 31)) & 1u);  // (one word per 64 lanes: one request)
  const int o = idx * 3;
  const int k = o & 3;
  // The next stone's vectors are needed only if pass 1 can advance the index at all (ENV:433-441: the reach counter is
  // one short of stop_frames) -- known from the state word alone, before any contact data: most envs fetch the 12 bytes
  // of the current stone only, which straddle a 64-byte fill boundary half as often as the 24 bytes of both stones.
  const bool has_next = idx < a.num_stones - 1 && state_count(word) + 1 >= a.stop_frames;
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f), l = r, r2 = r, l2 = r;
  const uint64_t once = policy_evict_first(), keep = policy_evict_last();
  if (live) {
    const float4* rrow = reinterpret_cast<const float4*>(in.contact_right + e * in.contact_right_stride) + (o >> 2);
    const float4* lrow = reinterpret_cast<const float4*>(in.contact_left + e * in.contact_left_stride) + (o >> 2);
    if (!a.lean) {
      // chunk 1 is needed unless the row ends with this stone's vector (idx = S-1 has k = 1: inside chunk 0)
      if (half == 0 || has_next || k >= 2) {
        r = ldg64_once_f4(rrow + half, once);
        l = ldg64_once_f4(lrow + half, once);
      }
      if (half == 0 && k == 3 && has_next) {  // floats 3..8: the tail of the second vector sits in a third chunk
        r2 = ldg64_once_f4(rrow + 2, once);
        l2 = ldg64_once_f4(lrow + 2, once);
      }
    } else if (half == 0 || k >= 2) {  // lean: the current stone's vector only -- one request per foot (.z/.w unused)
      r = ldg64_f4(rrow + half);
      l = ldg64_f4(lrow + half);
    }
  }
  // the six floats as f[k .. k+5] of the concatenation chunk0 (even lane) | chunk1 (odd lane) | chunk2 (even lane)
  float rc[12], lc[12];
  rc[0] = r.x; rc[1] = r.y; rc[2] = r.z; rc[3] = r.w;
  lc[0] = l.x; lc[1] = l.y; lc[2] = l.z; lc[3] = l.w;
  rc[4] = __shfl_down_sync(0xffffffffu, r.x, 1); rc[5] = __shfl_down_sync(0xffffffffu, r.y, 1);
  rc[6] = __shfl_down_sync(0xffffffffu, r.z, 1); rc[7] = __shfl_down_sync(0xffffffffu, r.w, 1);
  lc[4] = __shfl_down_sync(0xffffffffu, l.x, 1); lc[5] = __shfl_down_sync(0xffffffffu, l.y, 1);
  lc[6] = __shfl_down_sync(0xffffffffu, l.z, 1); lc[7] = __shfl_down_sync(0xffffffffu, l.w, 1);
  rc[8] = r2.x; rc[9] = 0.f; rc[10] = 0.f; rc[11] = 0.f;
  lc[8] = l2.x; lc[9] = 0.f; lc[10] = 0.f; lc[11] = 0.f;
  if (live) {
    if (stale) {  // lane h rewrites entries 2h, 2h+1 of the record
      refresh_window_entry(a.ws, e, idx, 2 * half, a.num_stones);
      refresh_window_entry(a.ws, e, idx, 2 * half + 1, a.num_stones);
    }
    if (a.body_dense) {  // even lane: the two feet, odd lane: the torso
      const int b0 = half ? 2 : 0, b1 = half ? 3 : 2;
      for (int b = b0; b < b1; ++b) {
        const int row = b == 0 ? in.right_foot_row : (b == 1 ? in.left_foot_row : in.torso_row);
        const float* src = in.body_pos + e * in.body_env_stride + row * in.body_row_stride;
#pragma unroll
        for (int c = 0; c < 3; ++c) a.body_dense[e * 9 + b * 3 + c] = ldg64_f(src + c);
      }
    }
  }
  if (!live || half) return;
  float v[6], u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {  // select by k without dynamic indexing of the register arrays
    v[i] = k == 0 ? rc[i] : (k == 1 ? rc[i + 1] : (k == 2 ? rc[i + 2] : rc[i + 3]));
    u[i] = k == 0 ? lc[i] : (k == 1 ? lc[i + 1] : (k == 2 ? lc[i + 2] : lc[i + 3]));
  }
  const float f_r = norm3(v[0], v[1], v[2]), f_l = norm3(u[0], u[1], u[2]);  // ENV:421-424
  const float f_r2 = has_next ? norm3(v[3], v[4], v[5]) : f_r;
  const float f_l2 = has_next ? norm3(u[3], u[4], u[5]) : f_l;
  // ENV:425 evaluated here: four bits per env instead of four floats (16 -> 1 byte written here and read by the step)
  const float eps = a.contact_epsilon;
  st_keep_u8(a.ws.contact_pre + e, (f_r > eps ? 1u : 0u) | (f_l > eps ? 2u : 0u) | (f_r2 > eps ? 4u : 0u) | (f_l2 > eps ? 8u : 0u),
             keep);  // read by the step kernel in a moment
}

#ifndef AS_STEP_MIN_CTAS
#define AS_STEP_MIN_CTAS (512 / AS_KTILE)
#endif
// FULL = true: the grid covers the full tiles; FULL = false: a one-CTA launch for the ragged last tile (tile_base =
// its index).  Two kernels, not a branch in one: compiled together, the ragged instantiation more than doubles the
// code and its register needs leak into the allocation of the hot one (ptxas: 246 instead of 56 spilled bytes).
template <int MODE, int EXACT, bool FULL, bool FAST = false, bool PACKED = false, bool PRE = false>
__global__ void __launch_bounds__(kThreads, AS_STEP_MIN_CTAS) k_step(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  Misc* misc = reinterpret_cast<Misc*>(smem + kOffMisc);
  // lets a kernel launched as a programmatic dependent (k_fixup_finish) become resident once every CTA of this grid
  // has started; it still waits for this grid to complete before touching memory.  No effect otherwise.
  if (MODE == kModeFused) asm volatile("griddepcontrol.launch_dependents;");
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&misc->mbar_root), 1);
    mbar_init(smem_u32(&misc->mbar_joint), 1);
  }
  if (MODE == kModeFused && threadIdx.x < 32) {
    ResetTables& T = misc->rt;
    const int l = threadIdx.x;
    load_reset_tables(a.P, a.jc, l, T.jc[l], T.pose[l], T.pose_mirrored[l], T.vel_mirrored[l]);
  }
  __syncthreads();
  uint32_t phase_root = 0, phase_joint = 0;
  const int tile = FULL ? static_cast<int>(blockIdx.x) : a.tile_base;  // (full tiles start at 0; the ragged launch is one CTA)
  static_assert(!PACKED || FULL, "a packed root tile needs a full tile (its byte count must be a multiple of 16)");
  static_assert(!PRE || (FULL && (MODE == kModeFused || MODE == kModePass1)), "the prepared path needs full tiles");
  process_tile<MODE, FULL, EXACT, FAST, PACKED, PRE>(a, tile, phase_root, phase_joint, smem);
}

// as_fold_stats: fold early so that the caller can all-reduce the statistics before as_finish_step.  One warp.  At most
// once per step: when the step closed itself, or its last CTA folded for the peer exchange, the totals are in
// ctrl->stats already and the slots are empty.
__global__ void __launch_bounds__(32) k_fold_early(Ctrl* ctrl, int64_t num_envs) {
  if (__ldcg(&ctrl->step_state) == 2u || __ldcg(&ctrl->stats_folded) != 0u) return;
  fold_stats_warp(ctrl, num_envs, threadIdx.x);
  if (threadIdx.x == 0) ctrl->stats_folded = 1;
}

// What a k_peer_exchange launch closes.
enum ExchangeMode {
  kExchangeFused = 0,  // behind k_step<fused>: fold this step's counters first; k_fixup_finish closes on the sums
  kExchangePass1 = 1,  // global 3-call mode, behind k_step<pass1> (whose last CTA folded already)
  kExchangeReset = 2,  // global 3-call mode, behind k_prepare_reset: `_reset_idx` outside a step, entered on every rank
};

// Fold + cross-shard sum in one kernel over NVLink peer memory (replaces k_fold_early + NCCL all-reduce of 80 bytes).
// One CTA.  Lane r of warp 0 talks to rank r: it stores this shard's ten counters into OUR slot of rank r's buffer,
// fences, then stores the epoch as the flag; it then polls rank r's slot in OUR buffer for the same epoch and reads
// the counters.  Two slots per sender (epoch parity): a rank can run at most one step ahead of a peer that has not
// yet read, because it cannot close step t+1 without that peer's step-t+1 counters.
// In the global 3-call modes the exchange also decides what needs all shards before `_reset_idx` runs: the promotion
// of ENV:471 on the global sums, "did any env reset" (DRL:359-360), and it adds the grid outcomes still pending from
// the previous step (summed over the shards) to the histograms, before anything draws from them.
__global__ void __launch_bounds__(128) k_peer_exchange(Ctrl* ctrl, const __grid_constant__ PeerArgs peer,
                                                       int64_t num_envs, int grid_cells,
                                                       const __grid_constant__ AsParams P, int mode) {
  __shared__ unsigned int s_timeouts;
  asm volatile("griddepcontrol.launch_dependents;");  // the finish kernel may become resident; it waits for us
  asm volatile("griddepcontrol.wait;" ::: "memory");  // the step kernel has completed and flushed
  const int tid = threadIdx.x;
  if (mode == kExchangeFused) {
    if (tid < 32 && __ldcg(&ctrl->stats_folded) == 0u) fold_stats_warp(ctrl, num_envs, tid);  // (unless as_fold_stats did)
    if (tid == 0) ctrl->stats_folded = 1;
    __syncthreads();
  }
  const unsigned long long epoch = static_cast<unsigned long long>(ctrl->peer_epoch) + 1ull;
  const int par = static_cast<int>(epoch & 1ull);
  auto grid_slot = [&](int owner, int sender) {
    return reinterpret_cast<PeerGrid*>(reinterpret_cast<unsigned char*>(peer.buf[owner]) + kPeerGridOffset) +
           par * kMaxPeers + sender;
  };
  if (grid_cells > 0) {
    // this step's difficulty-grid outcomes go first (all threads), the flag that publishes them last (below)
    for (int r = 0; r < peer.world; ++r) {
      PeerGrid* dst = grid_slot(r, peer.rank);
      for (int i = tid; i < grid_cells; i += blockDim.x) {
        asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(&dst->att[i]), "r"(ctrl->grid_delta_att[i]) : "memory");
        asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(&dst->succ[i]), "r"(ctrl->grid_delta_succ[i]) : "memory");
      }
    }
    __threadfence_system();
    __syncthreads();
  }
  if (tid < 32) {
    long long got[kPeerCounters];
    unsigned long long ep;
    const unsigned n_to = peer_sum_counters_warp(ctrl, peer, tid, got, ep);
    if (tid == 0) {
      s_timeouts = n_to;
      peer_publish(ctrl, peer, got, n_to, ep);
    }
  }
  __syncthreads();  // every peer's flag has been seen (acquire) by a lane of warp 0: their grid records are readable
  if (grid_cells > 0) {
    const bool ok = s_timeouts == 0;
    for (int i = tid; i < kMaxGridBins; i += blockDim.x) {
      unsigned int att = 0, succ = 0;
      if (i < grid_cells) {
        if (ok) {
          for (int r = 0; r < peer.world; ++r) {
            const PeerGrid* src = grid_slot(peer.rank, r);
            unsigned int x, y;
            asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(x) : "l"(&src->att[i]) : "memory");
            asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(y) : "l"(&src->succ[i]) : "memory");
            att += x;
            succ += y;
          }
        } else {
          att = ctrl->grid_delta_att[i];
          succ = ctrl->grid_delta_succ[i];
        }
      }
      ctrl->gx.grid_attempts[i] = att;
      ctrl->gx.grid_successes[i] = succ;
      if (mode != kExchangeFused && i < grid_cells) {  // the previous step's outcomes of all shards join the histograms
        grid_fold(ctrl->grid_attempts[i], ctrl->grid_successes[i], att, succ);
        ctrl->grid_delta_att[i] = ctrl->grid_delta_succ[i] = 0u;
      }
    }
  }
  if (mode != kExchangeFused && tid == 0) {
    AsStats g = ctrl->gx.stats;  // (this shard's own record if a peer timed out)
    if (mode == kExchangeReset) g.n_reset = 1;
    ctrl->promote_cur = promotion_decision(P, g);  // in force from here on; k_reset_list does not decide again
    ctrl->any_reset = g.n_reset > 0 ? 1u : 0u;
  }
}

// Fix-up + finish.  If NO env of this shard reset, the reference never runs pass 2 (DRL:360): redo every tile
// without it from the untouched pre-step state buffer (rare: needs zero resets among all envs).  The LAST CTA to
// have taken that decision (and done its share of the fix-up, if any) then folds the statistics, publishes next
// step's promotion, flips the state parity and advances the Philox step counter.  It has to be the last one: the
// finisher rewrites exactly the words the decision is read from (the counter slots, stats_folded), so nobody may
// still be about to read them.
__global__ void __launch_bounds__(kThreads, 2) k_fixup_finish(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  Misc* misc = reinterpret_cast<Misc*>(smem + kOffMisc);
  Ctrl* ctrl = a.ws.ctrl;
  const int tid = threadIdx.x;
  asm volatile("griddepcontrol.wait;" ::: "memory");  // (returns at once unless launched as a programmatic dependent)
  if (__ldcg(&ctrl->step_state) == 2u) return;  // the step kernel's last CTA closed the step itself (the common case)
  const bool prefolded = ctrl->stats_folded != 0;  // as_fold_stats ran: the slots are empty, the totals are in stats
  if (tid < 32) {
    // "did any env reset" (DRL:359-360) is a property of ALL envs: with a global sum at hand, that one decides
    unsigned n;
    if (a.global_stats) n = a.global_stats->stats.n_reset > 0 ? 1u : 0u;
    else n = prefolded ? static_cast<unsigned>(ctrl->stats.n_reset) : slot_sum(ctrl, kCntReset);
    if (tid == 0) misc->is_last = n;  // reused as "number of resets this step"
  }
  if (tid == 0) {
    mbar_init(smem_u32(&misc->mbar_root), 1);
    mbar_init(smem_u32(&misc->mbar_joint), 1);
  }
  __syncthreads();
  const bool need_fixup = misc->is_last == 0 && !(a.P.flags & AS_FLAG_SKIP_PASS2);
  __syncthreads();
  if (need_fixup) {
    uint32_t phase_root = 0, phase_joint = 0;
    for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
      process_tile<kModeFixup, false, 2>(a, tile, phase_root, phase_joint, smem);
      __syncthreads();
    }
    __threadfence();
    __syncthreads();
  }
  if (tid == 0) {
    const unsigned t = atomicAdd(&ctrl->blocks_done2, 1u);
    misc->is_last = (t == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (misc->is_last == 0) return;
  __threadfence();
  if (!prefolded && tid < 32) fold_stats_warp(ctrl, a.num_envs, tid);
  if (a.P.flags & AS_FLAG_GRID_CURRICULUM) {
    // this step's episode outcomes join the difficulty-grid histograms (the sum over all shards when one was handed in)
    for (int i = tid; i < kMaxGridBins; i += blockDim.x) {
      grid_fold(ctrl->grid_attempts[i], ctrl->grid_successes[i],
                a.global_stats ? a.global_stats->grid_attempts[i] : ctrl->grid_delta_att[i],
                a.global_stats ? a.global_stats->grid_successes[i] : ctrl->grid_delta_succ[i]);
    }
    __syncthreads();
    for (int i = tid; i < kMaxGridBins; i += blockDim.x) ctrl->grid_delta_att[i] = ctrl->grid_delta_succ[i] = 0u;
  }
  if (tid == 0) {
    close_step(a, ctrl, a.global_stats ? a.global_stats->stats : ctrl->stats, static_cast<unsigned>(ctrl->stats.n_reset));
    ctrl->blocks_done2 = 0;
    if (need_fixup) {
      ctrl->fixup_ran += 1;
      ctrl->stats.n_advanced -= ctrl->last_adv2;  // pass-2 advances were discarded with pass 2
    }
  }
}

}  // namespace as
