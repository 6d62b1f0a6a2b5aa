// C ABI of the B200-native Allsteps-v0 MDP step (include/allsteps_b200.h): argument checking, launch geometry,
// and nothing else.  All arithmetic lives in the kernels (as_step_kernel.cuh, as_aux_kernels.cuh).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

#include "as_aux_kernels.cuh"

using namespace as;

struct AsHandle {
  AsParams params;
  int64_t num_envs;
  int64_t env_id_offset;
  int device;
  int sm_count;
  Workspace ws;
  int64_t launches;
  MirrorTable mirror_obs, mirror_act;
  JointConsts jc;
  float inv_step_dt;
  float obs_clip_pass1;  // AsStepOut.obs_clip of the last as_step_pass1 (applied by as_step_pass2 too)
  int pdl;             // programmatic dependent launch: >= 1 k_fixup_finish after the step kernel, >= 2 also the step
                       // kernel after the gather kernel (ALLSTEPS_PDL, default 2; 0 = plain stream order)
  const void* lean_probe_ptr;  // last contact matrix whose memory type was looked up (pinned host => lean k_prepare)
  bool lean_probe_host;
  int regen_mode;      // shape of the regeneration kernel: 0 = by list length, 1 = warp per env, 2 = thread per env (ALLSTEPS_REGEN_MODE)
  cudaEvent_t ev_start, ev_stop;  // optional timing hook around k_step<fused>
  PeerArgs peer;        // world > 0 after as_peer_create; buf[] complete after as_peer_connect
  bool peer_connected;
  bool peer_three_call; // as_peer_three_call: the 3-call path decides promotion, any-reset and histograms over all shards
  volatile uint32_t* peer_host_error;  // mapped pinned host word the exchange kernel sets when a peer timed out
  bool pass1_done;
  bool device_list;     // as_reset took the envs from the list pass 1 compacted on the device (no host round trip)
  bool spec_valid;      // as_step_pass1 speculated pass 2 into the other state buffer; as_step_pass2 / as_step_no_reset closes it
  float* spec_obs;      // the observation buffer that pass 1 wrote
  bool pending_valid;   // a fused step was launched and still needs as_finish_step
  StepArgs pending;     // its arguments: the conditional fix-up re-reads the same inputs
};

namespace {

thread_local std::string g_error;

int fail(int code, const std::string& msg) {
  g_error = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_error = std::string(what) + ": " + cudaGetErrorString(e);
  return AS_ERR_CUDA;
}
#define AS_CUDA(call)                                   \
  do {                                                  \
    cudaError_t _e = (call);                            \
    if (_e != cudaSuccess) return cuda_fail(_e, #call); \
  } while (0)
#define AS_REQUIRE(cond, msg) \
  do {                        \
    if (!(cond)) return fail(AS_ERR_INVALID, msg); \
  } while (0)

int check_launch(AsHandle* h, const char* what) {
  h->launches += 1;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, what);
  return AS_OK;
}

// A peer exchange that timed out is fatal and sticky (the shards may have decided the promotion rule on different
// sums): the exchange kernel raised the mapped host word, every later step is refused.  A plain host read, no sync.
int check_peer(const AsHandle* h) {
  if (h->peer_host_error && *h->peer_host_error != 0u) {
    return fail(AS_ERR_PEER, "peer exchange timed out at epoch " + std::to_string(*h->peer_host_error & 0x7FFFFFFFu) +
                                 ": a shard did not deliver its step counters in time; the shards may have diverged");
  }
  return AS_OK;
}

int num_tiles(int64_t n) { return static_cast<int>((n + kTile - 1) / kTile); }

// AsParams.num_steps as the kernels take it: 0 means the default course length; -1 when out of range
int course_length(const AsParams& P) {
  const int S = P.num_steps == 0 ? kS : static_cast<int>(P.num_steps);
  return P.num_steps <= AS_MAX_STONES && S >= AS_MIN_STONES ? S : -1;
}
int handle_stones(const AsHandle* h) { return static_cast<int>(h->params.num_steps); }

constexpr int64_t kRegenByWarpMaxEnvs = 1 << 15;  // k_reset_rows: a warp per env up to this batch size (profiles/r02_experiments.txt, 12)
// From this batch size on the scattered reads of a step go to k_prepare*.  Below it the step is launch-latency bound
// (working set in L2, a handful of CTAs per SM): one launch fewer beats the better latency hiding of the separate gather
// kernel (measured, us per step with / without k_prepare*: 32 768 envs 22.1 / 22.0, 65 536 envs 25.9 / 27.6,
// 131 072 envs 40.9 / 47.5, 524 288 envs 107 / 130).
constexpr int64_t kSeparateGatherMinEnvs = 1 << 16;

// Contact matrices in pinned host memory (zero-copy ingest): every load of the gather is a PCIe request, so k_prepare*
// fetches the current stone's vectors only and the step kernel instantiation with its own gathers is used.
bool contact_in_host_memory(AsHandle* h, const AsStateIn* in) {
  if (in->contact_right != h->lean_probe_ptr) {
    cudaPointerAttributes attr;
    const cudaError_t e = cudaPointerGetAttributes(&attr, in->contact_right);
    h->lean_probe_host = e == cudaSuccess && attr.type == cudaMemoryTypeHost;
    if (e != cudaSuccess) cudaGetLastError();
    h->lean_probe_ptr = in->contact_right;
  }
  return h->lean_probe_host;
}

// k_prepare*: contact norms of the current / following stone, stale stone windows, optionally the three body rows out
// of a strided body tensor (`gather_body`), for batches that are not launch-bound.
int launch_prepare(AsHandle* h, const AsStateIn* in, cudaStream_t s, bool gather_body) {
  if (h->num_envs < kSeparateGatherMinEnvs) return AS_OK;
  PrepareArgs p;
  p.in = *in;
  p.ws = h->ws;
  p.num_envs = h->num_envs;
  p.body_dense = gather_body ? h->ws.body_dense : nullptr;
  p.lean = contact_in_host_memory(h, in) ? 1 : 0;
  p.stop_frames = h->params.stop_frames;
  p.contact_epsilon = h->params.contact_epsilon;
  p.num_stones = handle_stones(h);
  const bool aligned = ((reinterpret_cast<uintptr_t>(in->contact_right) | reinterpret_cast<uintptr_t>(in->contact_left)) &
                        15u) == 0 && ((in->contact_right_stride | in->contact_left_stride) & 3) == 0;
  if (aligned) {  // two lanes per env: one memory request per force vector
    const unsigned blocks = static_cast<unsigned>((2 * h->num_envs + 255) / 256);
    k_prepare_paired<<<blocks, 256, 0, s>>>(p);
    return check_launch(h, "k_prepare_paired");
  }
  const unsigned blocks = static_cast<unsigned>((h->num_envs + 255) / 256);
  k_prepare<<<blocks, 256, 0, s>>>(p);
  return check_launch(h, "k_prepare");
}

// AsStepOut.final_obs: optional, a full-size (N,59) buffer of its own (the kernels write its rows while the
// observation tile goes to obs)
int validate_final_obs(const AsHandle* h, const AsStepOut* out) {
  if (!out->final_obs) return AS_OK;
  const uintptr_t f = reinterpret_cast<uintptr_t>(out->final_obs);
  const uintptr_t o = reinterpret_cast<uintptr_t>(out->obs);
  const uintptr_t bytes = static_cast<uintptr_t>(h->num_envs) * kObs * sizeof(float);
  AS_REQUIRE((f & 3u) == 0, "final_obs must be 4-byte aligned");
  AS_REQUIRE(f + bytes <= o || o + bytes <= f, "final_obs must not overlap obs");
  return AS_OK;
}

int validate_state_in(const AsHandle* h, const AsStateIn* in, bool need_origins) {
  AS_REQUIRE(in != nullptr, "AsStateIn is null");
  AS_REQUIRE(in->root_pos && in->root_quat && in->root_lin_vel, "root state pointers must be set");
  AS_REQUIRE(in->body_pos, "body_pos must be set");
  AS_REQUIRE(in->joint_pos && in->joint_vel, "joint state pointers must be set");
  AS_REQUIRE(in->contact_right && in->contact_left, "contact matrices must be set");
  AS_REQUIRE(in->root_pos_stride >= 3 && in->root_quat_stride >= 4 && in->root_lin_vel_stride >= 3,
             "root strides too small");
  AS_REQUIRE(in->joint_pos_stride >= kJ && in->joint_vel_stride >= kJ, "joint strides too small");
  const int S = handle_stones(h);
  AS_REQUIRE(in->contact_right_stride >= S * 3 && in->contact_left_stride >= S * 3, "contact strides too small");
  AS_REQUIRE(in->body_row_stride >= 3 && in->body_env_stride >= 3, "body strides too small");
  AS_REQUIRE(in->right_foot_row >= 0 && in->left_foot_row >= 0 && in->torso_row >= 0, "negative body row");
  if (need_origins) AS_REQUIRE(in->env_origins != nullptr, "env_origins must be set for the fused step");
  return AS_OK;
}

void build_mirror_tables(AsHandle* h) {
  // ENV:574-584: swap right/left joint columns (+ their velocity columns and the two contact flags), negate
  // roll, v_y, the negation joints (pos and vel) and the y of the three stone targets.
  const AsParams& P = h->params;
  MirrorTable& o = h->mirror_obs;
  o.dim = kObs;
  for (int c = 0; c < kObs; ++c) {
    o.src[c] = c;
    o.sign[c] = 1.0f;
  }
  MirrorTable& a = h->mirror_act;
  a.dim = kJ;
  for (int c = 0; c < kObs; ++c) {
    a.src[c] = c < kJ ? c : 0;
    a.sign[c] = 1.0f;
  }
  for (int j = 0; j < kJ; ++j) {
    const int s = P.mirror_src[j];
    a.src[j] = s;
    a.sign[j] = P.mirror_sign[j];
    o.src[6 + j] = 6 + s;
    o.src[6 + kJ + j] = 6 + kJ + s;
    o.sign[6 + j] = P.mirror_sign[j];
    o.sign[6 + kJ + j] = P.mirror_sign[j];
  }
  o.src[48] = 49;
  o.src[49] = 48;
  o.sign[1] = -1.0f;
  o.sign[4] = -1.0f;
  o.sign[51] = o.sign[54] = o.sign[57] = -1.0f;
}

// Correctly rounded fp32 reciprocal of d (needed by the two-FMA quotient in scale_joint).
float rn_reciprocal(float d) {
  float best = static_cast<float>(1.0 / static_cast<double>(d));
  double best_err = std::fabs(1.0 - static_cast<double>(best) * static_cast<double>(d));  // product is exact
  const float cands[2] = {std::nextafterf(best, 0.0f), std::nextafterf(best, 2.0f * best)};
  for (float c : cands) {
    const double err = std::fabs(1.0 - static_cast<double>(c) * static_cast<double>(d));
    if (err < best_err) {
      best = c;
      best_err = err;
    }
  }
  return best;
}

void build_joint_consts(AsHandle* h) {
  const AsParams& P = h->params;
  JointConsts& c = h->jc;
  c.exact_div = 0;
  for (int j = 0; j < kJ; ++j) {
    // same fp32 roundings as MATH:36-40: offset = (lower + upper) * 0.5 ; denominator = upper - lower
    volatile float sum = P.joint_lower[j] + P.joint_upper[j];
    volatile float range = P.joint_upper[j] - P.joint_lower[j];
    c.c[j] = make_float4(sum * 0.5f, range * 0.5f, 2.0f * rn_reciprocal(range), 0.99f);  // (the factors 2 are exact)
    uint32_t bits;
    const float r = range;
    std::memcpy(&bits, &r, sizeof(bits));
    if ((bits & 0x7FFFFFu) == 0x7FFFFFu) c.exact_div = 1;  // Markstein's excluded case
  }
  uint32_t dt_bits;
  std::memcpy(&dt_bits, &P.step_dt, sizeof(dt_bits));
  if ((dt_bits & 0x7FFFFFu) == 0x7FFFFFu) c.exact_div = 1;  // the same for the divisor of ENV:416
  h->inv_step_dt = rn_reciprocal(P.step_dt);
}

StepArgs make_step_args(AsHandle* h, const AsStateIn* in, const float* actions, int64_t actions_stride,
                        const AsStepOut* out) {
  StepArgs a;
  std::memset(&a, 0, sizeof(a));
  a.P = h->params;
  a.jc = h->jc;
  a.inv_step_dt = h->inv_step_dt;
  if (in) a.in = *in;
  a.actions = actions;
  a.actions_stride = actions_stride;
  if (out) a.out = *out;
  a.ws = h->ws;
  a.num_envs = h->num_envs;
  a.env_id_offset = h->env_id_offset;
  a.num_tiles = num_tiles(h->num_envs);
  // which views the TMA engine can take: dense rows and a 16-byte aligned base (tiles start every 128 rows)
  auto dense = [](const void* p, int64_t stride, int64_t width) {
    return p != nullptr && stride == width && (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
  };
  uint32_t bits = 0;
  if (in) {
    if (dense(in->joint_pos, in->joint_pos_stride, kJ)) bits |= kDenseJp;
    if (dense(in->joint_vel, in->joint_vel_stride, kJ)) bits |= kDenseJv;
    if (dense(in->root_pos, in->root_pos_stride, 3)) bits |= kDenseRp;
    if (dense(in->root_quat, in->root_quat_stride, 4)) bits |= kDenseRq;
    if (dense(in->root_lin_vel, in->root_lin_vel_stride, 3)) bits |= kDenseRv;
    if (in->body_row_stride == 3 && in->right_foot_row == 0 && in->left_foot_row == 1 && in->torso_row == 2 &&
        dense(in->body_pos, in->body_env_stride, 9))
      bits |= kDenseBody;
    if (dense(in->env_origins, 3, 3)) bits |= kDenseOrg;
  }
  if (dense(actions, actions_stride, kJ)) bits |= kDenseAct;
  if (out && dense(out->obs, kObs, kObs)) bits |= kDenseObs;
  a.dense16 = bits;
  a.use_pre = h->num_envs >= kSeparateGatherMinEnvs ? 1 : 0;
  return a;
}

ResetArgs make_reset_args(AsHandle* h, const float* env_origins) {
  ResetArgs r;
  std::memset(&r, 0, sizeof(r));
  r.P = h->params;
  r.ws = h->ws;
  r.env_origins = env_origins;
  r.num_envs = h->num_envs;
  r.env_id_offset = h->env_id_offset;
  return r;
}

int grid_for(int64_t items, int per_block, int sm_count, int max_waves) {
  int64_t blocks = (items + per_block - 1) / per_block;
  const int64_t cap = static_cast<int64_t>(sm_count) * max_waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

// A kernel launch that may start under the tail of the kernel before it in the stream (programmatic dependent launch).
template <typename... KArgs, typename... Args>
cudaError_t launch_dependent(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s,
                             bool programmatic, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = programmatic ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// k_reset_rows over the list of envs that regenerate (Ctrl::n_regen_list), behind the kernel that compacted it: the
// fused step kernel or k_reset_list.  Shape: a warp per env for small batches, a thread per env for large ones
// (ALLSTEPS_REGEN_MODE: 1 / 2).
int launch_regeneration(AsHandle* h, const ResetArgs& r, cudaStream_t s) {
  const bool by_warp = h->regen_mode == 1 || (h->regen_mode == 0 && h->num_envs <= kRegenByWarpMaxEnvs);
  const bool default_s = handle_stones(h) == kS;
  const int grid_ctas = grid_for(h->num_envs, 64, h->sm_count, 8);
  AS_CUDA(launch_dependent(by_warp ? (default_s ? k_reset_rows<true, true> : k_reset_rows<true, false>)
                                   : (default_s ? k_reset_rows<false, true> : k_reset_rows<false, false>),
                           static_cast<unsigned>(grid_ctas), 256u, 0, s, h->pdl >= 1, r));
  return check_launch(h, "k_reset_rows");
}

// k_peer_exchange behind the kernel just launched (ExchangeMode: what it closes).
int launch_exchange(AsHandle* h, int mode, cudaStream_t s) {
  const int cells = (h->params.flags & AS_FLAG_GRID_CURRICULUM) ? static_cast<int>(h->params.grid_bins * h->params.grid_bins) : 0;
  AS_CUDA(launch_dependent(k_peer_exchange, 1u, 128u, 0, s, h->pdl >= 1, h->ws.ctrl, h->peer, h->num_envs, cells,
                           h->params, mode));
  return check_launch(h, "k_peer_exchange");
}

using StepKernel = void (*)(StepArgs);

// The families of k_step instantiations (process_tile describes FAST, PACKED and PRE).
enum StepKind {
  kRagged,      // the one-CTA launch of a ragged last tile; division flavour read at run time (EXACT = 2)
  kRuntimeDiv,  // full tiles, division flavour read at run time: pass 2, true divisions, pass 1 not prepared
  kTwoFma,      // full tiles of a fused step that gathers its contact vectors itself, two-FMA quotients; FAST / PACKED
  kPrepared,    // full tiles behind k_prepare*, two-FMA quotients (PRE); FAST / PACKED variants
};

// Every k_step instantiation the library launches.  select_step picks from this table alone and as_create sets the
// dynamic shared-memory limit of every entry, so whatever can be selected can be launched.
struct StepVariant {
  int mode;  // StepMode
  StepKind kind;
  bool fast, packed;
  StepKernel kernel;
};
const StepVariant kStepVariants[] = {
    {kModeFused, kRagged, false, false, k_step<kModeFused, 2, false>},
    {kModeFused, kRuntimeDiv, false, false, k_step<kModeFused, 2, true>},
    {kModeFused, kTwoFma, false, false, k_step<kModeFused, 0, true, false, false>},
    {kModeFused, kTwoFma, false, true, k_step<kModeFused, 0, true, false, true>},
    {kModeFused, kTwoFma, true, false, k_step<kModeFused, 0, true, true, false>},
    {kModeFused, kTwoFma, true, true, k_step<kModeFused, 0, true, true, true>},
    {kModeFused, kPrepared, false, false, k_step<kModeFused, 0, true, false, false, true>},
    {kModeFused, kPrepared, false, true, k_step<kModeFused, 0, true, false, true, true>},
    {kModeFused, kPrepared, true, false, k_step<kModeFused, 0, true, true, false, true>},
    {kModeFused, kPrepared, true, true, k_step<kModeFused, 0, true, true, true, true>},
    {kModePass1, kRagged, false, false, k_step<kModePass1, 2, false>},
    {kModePass1, kRuntimeDiv, false, false, k_step<kModePass1, 2, true>},
    {kModePass1, kPrepared, false, false, k_step<kModePass1, 0, true, false, false, true>},
    {kModePass1, kPrepared, false, true, k_step<kModePass1, 0, true, false, true, true>},
    {kModePass1, kPrepared, true, false, k_step<kModePass1, 0, true, true, false, true>},
    {kModePass1, kPrepared, true, true, k_step<kModePass1, 0, true, true, true, true>},
    {kModePass2, kRagged, false, false, k_step<kModePass2, 2, false>},
    {kModePass2, kRuntimeDiv, false, false, k_step<kModePass2, 2, true>},
};

size_t step_smem(const StepVariant& v) { return v.packed ? kSmemBytesPacked : kSmemBytes; }

const StepVariant* find_step_variant(int mode, StepKind kind, bool fast, bool packed) {
  for (const StepVariant& v : kStepVariants)
    if (v.mode == mode && v.kind == kind && v.fast == fast && v.packed == packed) return &v;
  return nullptr;
}

struct StepLaunch {
  const StepVariant* full;
  const StepVariant* ragged;
};

// Chooses the k_step instantiations of a step in `mode` and sets what the kernel has to know about that choice in `a`.
StepLaunch select_step(AsHandle* h, int mode, const AsStateIn* in, StepArgs& a) {
  // pass 2 of the 3-call path outside a speculating pass 1 (a reset outside a step) is off the hot path: the generic
  // instantiation, in stream order, with the body rows read where they are
  const bool hot = mode != kModePass2;
  if (hot && a.use_pre && !(a.dense16 & kDenseBody)) {
    // The three body rows the task reads (12 bytes each out of Isaac Lab's (N,B,13) body_state_w) are scattered
    // reads like the contact vectors: k_prepare* gathers them into a dense (N,3,3) array, which the step kernel (and
    // the fix-up, which re-reads the inputs) then takes by bulk copy.
    a.body_from_prepare = 1;
    a.in.body_pos = h->ws.body_dense;
    a.in.body_env_stride = 9;
    a.in.body_row_stride = 3;
    a.in.right_foot_row = 0;
    a.in.left_foot_row = 1;
    a.in.torso_row = 2;
    a.dense16 |= kDenseBody;
  }
  // dependent of the gather kernel: tiles, state words and windows are loaded while the gather's last wave runs; the
  // MDP role waits for the gather (griddepcontrol.wait) right before it reads the contact norms.  Not between the timing
  // events of a fused step, which time the step kernel alone.
  a.pdl_wait = (hot && h->pdl >= 2 && a.use_pre && !(mode == kModeFused && h->ev_start)) ? 1 : 0;
  // the common launch shape has its own instantiation (process_tile: FAST)
  const bool fast = !a.in.quat_xyzw && !a.out.reward_terms && a.out.obs_clip == 0.0f && !a.out.final_obs &&
                    handle_stones(h) == kS;
  // root pos / quat / lin vel handed over as slices of one (N,13) root_state_w tensor (Isaac Lab's own layout): the
  // full tiles take the whole rows with one bulk copy (process_tile: PACKED)
  const bool packed = in->root_pos_stride == AS_ROOT_STATE_DIM && in->root_quat_stride == AS_ROOT_STATE_DIM &&
                      in->root_lin_vel_stride == AS_ROOT_STATE_DIM && in->root_quat == in->root_pos + 3 &&
                      in->root_lin_vel == in->root_pos + 7 && (reinterpret_cast<uintptr_t>(in->root_pos) & 15u) == 0;
  // (the host knows whether any divisor needs a true division: the two-FMA instantiations have no branch for it)
  StepKind kind = kRuntimeDiv;
  if (hot && !h->jc.exact_div && a.use_pre && !contact_in_host_memory(h, in)) kind = kPrepared;
  else if (mode == kModeFused && !h->jc.exact_div) kind = kTwoFma;
  const bool variants = kind != kRuntimeDiv;
  return {find_step_variant(mode, kind, variants && fast, variants && packed),
          find_step_variant(mode, kRagged, false, false)};
}

// Launches k_step over all tiles: a one-CTA launch of the ragged instantiation for a tail tile (first, so that in a
// programmatic chain the full-tile kernel, whose CTAs wait for their primary before they read the contact norms,
// cannot complete before it), then the full-tile instantiation.
cudaError_t launch_step(AsHandle* h, const StepLaunch& k, StepArgs& a, cudaStream_t s) {
  if (!k.full || !k.ragged) return cudaErrorInvalidDeviceFunction;  // (a combination missing from kStepVariants)
  const bool programmatic = a.pdl_wait != 0;
  const int n_full = static_cast<int>(a.num_envs / kTile);
  if (n_full < a.num_tiles) {
    a.tile_base = n_full;
    cudaError_t rc = launch_dependent(k.ragged->kernel, 1u, static_cast<unsigned>(kThreads), step_smem(*k.ragged), s,
                                      programmatic, a);
    if (rc != cudaSuccess) return rc;
    if (n_full > 0) h->launches += 1;  // (check_launch counts one launch per call)
  }
  a.tile_base = 0;
  if (n_full == 0) return cudaSuccess;
  return launch_dependent(k.full->kernel, static_cast<unsigned>(n_full), static_cast<unsigned>(kThreads),
                          step_smem(*k.full), s, programmatic, a);
}
}  // namespace

extern "C" {

int as_abi_version(void) { return AS_ABI_VERSION; }

const char* as_last_error(void) { return g_error.c_str(); }

int64_t as_workspace_bytes(int64_t num_envs) {
  if (num_envs <= 0) return 0;
  return workspace_layout(num_envs, kS).total;
}

int64_t as_workspace_bytes_for(const AsParams* params, int64_t num_envs) {
  if (!params || num_envs <= 0 || course_length(*params) < 0) return 0;
  return workspace_layout(num_envs, course_length(*params)).total;
}

int as_create(const AsParams* params, int64_t num_envs, int64_t env_id_offset, int device, void* workspace,
              int64_t workspace_bytes, void* stream, AsHandle** out) {
  AS_REQUIRE(params && out, "params/out is null");
  AS_REQUIRE(num_envs > 0 && num_envs < (1ll << 31), "num_envs out of range");
  AS_REQUIRE(env_id_offset >= 0 && env_id_offset + num_envs <= (1ll << 32), "global env ids must fit 32 bits");
  AS_REQUIRE(params->stop_frames >= 1 && params->stop_frames <= 3, "stop_frames must be in 1..3");
  AS_REQUIRE(params->max_level >= 0 && params->max_level < AS_NUM_LEVELS, "max_level out of range");
  AS_REQUIRE(params->max_episode_length > 1 && params->max_episode_length < kMaxEpisodeLength,
             "max_episode_length out of range");
  AS_REQUIRE(params->step_dt > 0.0f, "step_dt must be positive");
  const int S = course_length(*params);
  AS_REQUIRE(S > 0, "num_steps must be 0 (default) or in 3..32");
  if (params->flags & AS_FLAG_GRID_CURRICULUM)
    AS_REQUIRE(params->grid_bins >= 2 && params->grid_bins <= 16, "grid_bins must be in 2..16");
  for (int j = 0; j < kJ; ++j) {
    AS_REQUIRE(params->joint_upper[j] > params->joint_lower[j], "joint limits must satisfy lower < upper");
    AS_REQUIRE(params->mirror_src[j] >= 0 && params->mirror_src[j] < kJ, "mirror_src out of range");
  }
  const WorkspaceLayout l = workspace_layout(num_envs, S);
  AS_REQUIRE(workspace != nullptr && workspace_bytes >= l.total, "workspace too small (see as_workspace_bytes_for)");
  AS_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "workspace must be 256-byte aligned");
  AS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  AS_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    return fail(AS_ERR_CUDA, "this library contains sm_100a code only; device is sm_" + std::to_string(prop.major) +
                                 std::to_string(prop.minor));
  }
  // the step kernels stage more than the default 48 KB of dynamic shared memory
  for (const StepVariant& v : kStepVariants)
    AS_CUDA(cudaFuncSetAttribute(v.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(step_smem(v))));
  AS_CUDA(cudaFuncSetAttribute(k_fixup_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  AS_CUDA(cudaFuncSetAttribute(k_mirror_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, kMirrorSmemBytes));
  AsHandle* h = new (std::nothrow) AsHandle();
  AS_REQUIRE(h != nullptr, "out of host memory");
  h->params = *params;
  h->params.num_steps = static_cast<uint32_t>(S);  // (the kernels read the course length from here)
  h->num_envs = num_envs;
  h->env_id_offset = env_id_offset;
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->launches = 0;
  h->pass1_done = false;
  h->spec_valid = false;
  h->lean_probe_ptr = nullptr;
  h->lean_probe_host = false;
  h->device_list = false;
  h->spec_obs = nullptr;
  h->obs_clip_pass1 = 0.0f;
  std::memset(&h->peer, 0, sizeof(h->peer));
  h->peer_connected = false;
  h->peer_three_call = false;
  h->peer_host_error = nullptr;
  h->pending_valid = false;
  h->ev_start = h->ev_stop = nullptr;
  {
    const char* pdl = std::getenv("ALLSTEPS_PDL");
    h->pdl = pdl ? std::atoi(pdl) : 2;
    const char* rm = std::getenv("ALLSTEPS_REGEN_MODE");
    h->regen_mode = rm ? std::atoi(rm) : 0;
  }
  unsigned char* base = static_cast<unsigned char*>(workspace);
  h->ws.ctrl = reinterpret_cast<Ctrl*>(base + l.ctrl_off);
  h->ws.state[0] = reinterpret_cast<uint2*>(base + l.state0_off);
  h->ws.state[1] = reinterpret_cast<uint2*>(base + l.state1_off);
  h->ws.stones = reinterpret_cast<float4*>(base + l.stones_off);
  h->ws.window = reinterpret_cast<float4*>(base + l.window_off);
  h->ws.reset_ids = reinterpret_cast<int32_t*>(base + l.reset_ids_off);
  h->ws.regen_ids = reinterpret_cast<int32_t*>(base + l.regen_ids_off);
  h->ws.regen_info = reinterpret_cast<uint8_t*>(base + l.regen_info_off);
  h->ws.bin = reinterpret_cast<uint8_t*>(base + l.bin_off);
  h->ws.contact_pre = reinterpret_cast<uint8_t*>(base + l.contact_pre_off);
  h->ws.body_dense = reinterpret_cast<float*>(base + l.body_dense_off);
  h->ws.tail1 = reinterpret_cast<float4*>(base + l.tail1_off);
  h->ws.pass1_reset = reinterpret_cast<uint8_t*>(base + l.pass1_reset_off);
  h->ws.win_stale = reinterpret_cast<uint32_t*>(base + l.win_stale_off);
  build_mirror_tables(h);
  build_joint_consts(h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(workspace, 0, static_cast<size_t>(l.total), s);
  if (e != cudaSuccess) {
    delete h;
    return cuda_fail(e, "cudaMemsetAsync(workspace)");
  }
  // no stone window is valid yet (k_prepare* refreshes the records whose bit is set)
  e = cudaMemsetAsync(h->ws.win_stale, 0xFF, static_cast<size_t>((num_envs + 31) / 32 * 4), s);
  if (e != cudaSuccess) {
    delete h;
    return cuda_fail(e, "cudaMemsetAsync(win_stale)");
  }
  // initial MDP state of AllstepsEnv.__init__ (ENV:74-78): index 1, right leg swings, everything else zero -- in both
  // state buffers the packed word, which is nonzero in its lowest byte only
  const uint32_t word = pack_state(1, 0, 0, 0, 0);
  e = cudaMemset2DAsync(h->ws.state[0], 8, static_cast<int>(word & 0xFFu), 1, static_cast<size_t>(num_envs), s);
  if (e == cudaSuccess)
    e = cudaMemset2DAsync(h->ws.state[1], 8, static_cast<int>(word & 0xFFu), 1, static_cast<size_t>(num_envs), s);
  if (e != cudaSuccess) {
    delete h;
    return cuda_fail(e, "cudaMemset2DAsync(state)");
  }
  *out = h;
  return AS_OK;
}

void as_destroy(AsHandle* h) {
  if (!h) return;
  if (h->peer.world > 0) {
    cudaSetDevice(h->device);
    for (int r = 0; r < h->peer.world; ++r) {
      if (!h->peer.buf[r]) continue;
      if (r == h->peer.rank) cudaFree(h->peer.buf[r]);
      else cudaIpcCloseMemHandle(h->peer.buf[r]);
    }
    if (h->peer_host_error) cudaFreeHost(const_cast<uint32_t*>(h->peer_host_error));
  }
  delete h;
}

int as_generate_stones(AsHandle* h, const float* env_origins, const int32_t* env_ids, int64_t n_ids,
                       const float* uniforms, void* stream) {
  AS_REQUIRE(h && env_origins, "handle/env_origins is null");
  AS_REQUIRE(env_ids == nullptr || n_ids >= 0, "negative id count");
  ResetArgs r = make_reset_args(h, env_origins);
  r.env_ids = env_ids;
  r.n_ids = n_ids;
  r.stone_uniforms = uniforms;
  const int64_t n = env_ids ? n_ids : h->num_envs;
  if (n == 0) return AS_OK;
  const int grid = grid_for(n, 8, h->sm_count, 8);
  k_generate_stones<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(r);
  return check_launch(h, "k_generate_stones");
}

int as_step_fused(AsHandle* h, const AsStateIn* in, const float* actions, int64_t actions_stride,
                  const AsStepOut* out, const AsResetOut* reset_out, void* stream) {
  AS_REQUIRE(h && out && actions, "handle/out/actions is null");
  if (int rc = validate_state_in(h, in, true)) return rc;
  AS_REQUIRE(actions_stride >= kJ, "actions stride too small");
  AS_REQUIRE(out->obs && out->reward && out->terminated && out->time_out, "step outputs must be set");
  AS_REQUIRE(out->obs_clip >= 0.0f, "obs_clip must be >= 0");
  if (int rc = validate_final_obs(h, out)) return rc;
  if (h->pending_valid) return fail(AS_ERR_STATE, "previous fused step was not closed with as_finish_step");
  if (h->peer_three_call) return fail(AS_ERR_STATE, "the handle is in the global 3-call mode (as_peer_three_call)");
  if (int rc = check_peer(h)) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  StepArgs a = make_step_args(h, in, actions, actions_stride, out);
  const bool want_rows = reset_out && (reset_out->root_state || reset_out->joint_pos || reset_out->joint_vel ||
                                       reset_out->reset_ids || reset_out->n_reset);
  const bool grid = (h->params.flags & AS_FLAG_GRID_CURRICULUM) != 0;
  const bool regen_enabled = grid || (h->params.flags & AS_FLAG_INTENDED_REGEN) != 0;
  a.want_reset_list = (reset_out && reset_out->reset_ids) ? 1 : 0;
  if (want_rows) a.rows = *reset_out;  // start-pose rows are written by the step kernel itself
  const StepLaunch k = select_step(h, kModeFused, in, a);
  if (int rc = launch_prepare(h, in, s, a.body_from_prepare != 0)) return rc;
  if (h->ev_start) AS_CUDA(cudaEventRecord(h->ev_start, s));
  // the last CTA closes the step itself unless somebody else has to see the open step: the cross-shard exchange, an
  // all-reduce the caller announced (AS_STEP_DEFER_FINISH), or the regeneration kernels launched below
  a.self_finish = (!regen_enabled && !(out->flags & AS_STEP_DEFER_FINISH)) ? 1 : 0;
  if (h->peer_connected) a.peer = h->peer;  // (world > 0: the closing CTA sums the counters over the shards itself)
  AS_CUDA(launch_step(h, k, a, s));
  if (int rc = check_launch(h, "k_step<fused>")) return rc;
  if (h->ev_stop) AS_CUDA(cudaEventRecord(h->ev_stop, s));
  if (regen_enabled) {
    // kernels (b) + (c) over the compacted list: the grid curriculum's outcome record and new bins (sampled from the
    // histograms as they stand after the previous step; this step's outcomes join them when the step is closed) and
    // the stone rows.  A programmatic dependent of the step kernel: launch and prologue hide under its last wave.
    ResetArgs r = make_reset_args(h, in->env_origins);
    r.fused = 1;
    if (int rc = launch_regeneration(h, r, s)) return rc;
  }
  h->pending = a;
  h->pending_valid = true;
  return AS_OK;
}

int as_fold_stats(AsHandle* h, void* stream) {
  AS_REQUIRE(h, "handle is null");
  if (!h->pending_valid) return fail(AS_ERR_STATE, "as_fold_stats belongs between as_step_fused and as_finish_step");
  k_fold_early<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(h->ws.ctrl, h->num_envs);
  return check_launch(h, "k_fold_early");
}

int as_peer_create(AsHandle* h, int world, int rank, void* ipc_handle_out) {
  AS_REQUIRE(h && ipc_handle_out, "null argument");
  AS_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "world/rank out of range");
  AS_REQUIRE(h->peer.world == 0, "as_peer_create was already called on this handle");
  static_assert(sizeof(cudaIpcMemHandle_t) == AS_PEER_HANDLE_BYTES, "IPC handle size");
  AS_CUDA(cudaSetDevice(h->device));
  void* buf = nullptr;
  AS_CUDA(cudaMalloc(&buf, static_cast<size_t>(kPeerBufferBytes)));
  cudaError_t e = cudaMemset(buf, 0, static_cast<size_t>(kPeerBufferBytes));
  cudaIpcMemHandle_t ipc;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&ipc, buf);
  if (e != cudaSuccess) {
    cudaFree(buf);
    return cuda_fail(e, "peer buffer");
  }
  std::memcpy(ipc_handle_out, &ipc, sizeof(ipc));
  {
    void* host_word = nullptr;
    void* dev_view = nullptr;
    e = cudaHostAlloc(&host_word, 64, cudaHostAllocMapped);
    if (e == cudaSuccess) {
      std::memset(host_word, 0, 64);
      e = cudaHostGetDevicePointer(&dev_view, host_word, 0);
    }
    if (e != cudaSuccess) {
      if (host_word) cudaFreeHost(host_word);
      cudaFree(buf);
      return cuda_fail(e, "peer error word");
    }
    h->peer_host_error = static_cast<volatile uint32_t*>(host_word);
    h->peer.host_error = static_cast<uint32_t*>(dev_view);
    // how long the exchange kernel polls for a peer: ALLSTEPS_PEER_TIMEOUT_MS (default 10 s; 0 = without limit)
    const char* to = std::getenv("ALLSTEPS_PEER_TIMEOUT_MS");
    const long long ms = to ? std::atoll(to) : 10000;
    h->peer.timeout_ns = ms > 0 ? static_cast<unsigned long long>(ms) * 1000000ull : 0ull;
  }
  h->peer.world = world;
  h->peer.rank = rank;
  h->peer.buf[rank] = static_cast<PeerSlot*>(buf);
  h->peer_connected = false;
  return AS_OK;
}

int as_peer_connect(AsHandle* h, const void* ipc_handles_in_rank_order) {
  AS_REQUIRE(h && ipc_handles_in_rank_order, "null argument");
  AS_REQUIRE(h->peer.world > 0, "as_peer_connect without as_peer_create");
  AS_REQUIRE(!h->peer_connected, "peers are already connected");
  AS_CUDA(cudaSetDevice(h->device));
  const unsigned char* all = static_cast<const unsigned char*>(ipc_handles_in_rank_order);
  for (int r = 0; r < h->peer.world; ++r) {
    if (r == h->peer.rank) continue;
    cudaIpcMemHandle_t ipc;
    std::memcpy(&ipc, all + static_cast<size_t>(r) * AS_PEER_HANDLE_BYTES, sizeof(ipc));
    void* p = nullptr;
    AS_CUDA(cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
    h->peer.buf[r] = static_cast<PeerSlot*>(p);
  }
  h->peer_connected = true;
  return AS_OK;
}

int as_peer_three_call(AsHandle* h, int32_t enable) {
  AS_REQUIRE(h, "handle is null");
  if (!h->peer_connected) return fail(AS_ERR_STATE, "as_peer_three_call needs connected peers (as_peer_connect)");
  if (h->pending_valid || h->spec_valid) return fail(AS_ERR_STATE, "a step is open; switch the mode between steps");
  h->peer_three_call = enable != 0;
  return AS_OK;
}

int as_peer_status(AsHandle* h, int* world, int* rank, int64_t* timeouts, void* stream) {
  AS_REQUIRE(h, "handle is null");
  if (world) *world = h->peer_connected ? h->peer.world : 0;
  if (rank) *rank = h->peer.rank;
  if (timeouts) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned long long t = 0;
    AS_CUDA(cudaMemcpyAsync(&t, &h->ws.ctrl->peer_timeouts, sizeof(t), cudaMemcpyDeviceToHost, s));
    AS_CUDA(cudaStreamSynchronize(s));
    *timeouts = static_cast<int64_t>(t);
  }
  return AS_OK;
}

int as_global_stats_device_ptr(AsHandle* h, AsStats** device_stats) {
  AS_REQUIRE(h && device_stats, "null argument");
  *device_stats = &h->ws.ctrl->gx.stats;
  return AS_OK;
}

int as_exchange_device_ptr(AsHandle* h, AsExchange** local, AsExchange** global) {
  AS_REQUIRE(h, "handle is null");
  if (local) *local = reinterpret_cast<AsExchange*>(&h->ws.ctrl->stats);
  if (global) *global = &h->ws.ctrl->gx;
  return AS_OK;
}

int as_finish_step(AsHandle* h, const AsExchange* global_stats, void* stream) {
  AS_REQUIRE(h, "handle is null");
  if (!h->pending_valid) return fail(AS_ERR_STATE, "as_finish_step without a preceding as_step_fused");
  if (int rc = check_peer(h)) {
    h->pending_valid = false;
    return rc;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  StepArgs a = h->pending;  // the fix-up re-reads the inputs of the step it closes
  a.global_stats = global_stats;
  if (h->peer_connected && global_stats == nullptr && a.self_finish) {
    a.global_stats = &h->ws.ctrl->gx;  // the step kernel's last CTA exchanged the counters and (normally) closed the step
  } else if (h->peer_connected && global_stats == nullptr) {
    // fold + sum over the shards through NVLink peer memory, in one small kernel under the step kernel's tail
    if (int rc = launch_exchange(h, kExchangeFused, s)) return rc;
    a.global_stats = &h->ws.ctrl->gx;
  }
  const int grid = grid_for(a.num_tiles, 1, h->sm_count, 1);
  // programmatic dependent launch: the step kernel releases its dependents as soon as its last wave of CTAs is
  // resident, so this kernel's launch and prologue overlap that wave; it waits (griddepcontrol.wait) for the kernel
  // before it to complete and flush before it reads anything
  AS_CUDA(launch_dependent(k_fixup_finish, static_cast<unsigned>(grid), static_cast<unsigned>(kThreads), kSmemBytes, s,
                           h->pdl >= 1, a));
  h->pending_valid = false;
  return check_launch(h, "k_fixup_finish");
}

int as_step_pass1(AsHandle* h, const AsStateIn* in, const float* actions, int64_t actions_stride,
                  const int64_t* episode_length, const AsStepOut* out, void* stream) {
  AS_REQUIRE(h && out && actions, "handle/out/actions is null");
  if (int rc = validate_state_in(h, in, false)) return rc;
  AS_REQUIRE(actions_stride >= kJ, "actions stride too small");
  AS_REQUIRE(out->obs && out->reward && out->terminated && out->time_out, "step outputs must be set");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  AS_REQUIRE(out->obs_clip >= 0.0f, "obs_clip must be >= 0");
  if (int rc = validate_final_obs(h, out)) return rc;
  if (h->peer_three_call)
    if (int rc = check_peer(h)) return rc;
  StepArgs a = make_step_args(h, in, actions, actions_stride, out);
  a.ext_episode_length = episode_length;
  h->obs_clip_pass1 = out->obs_clip;  // as_step_pass2 rewrites the same observation buffer: same epilogue
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  AS_CUDA(cudaMemsetAsync(&h->ws.ctrl->n_reset_list, 0, sizeof(uint32_t), s));  // pass 1 compacts the flagged envs
  h->device_list = false;
  const StepLaunch k = select_step(h, kModePass1, in, a);
  if (int rc = launch_prepare(h, in, s, a.body_from_prepare != 0)) return rc;
  AS_CUDA(launch_step(h, k, a, s));
  h->pass1_done = true;   // (its last CTA folds the statistics and advances the Philox step counter)
  h->spec_valid = true;
  h->spec_obs = out->obs;
  if (int rc = check_launch(h, "k_step<pass1>")) return rc;
  // global 3-call mode: one exchange per step, right here -- everything the step needs from the other shards is known
  // (flagged count, sum of the indices), and so are the grid outcomes still pending from the previous step
  return h->peer_three_call ? launch_exchange(h, kExchangePass1, s) : AS_OK;
}

int as_reset(AsHandle* h, const float* env_origins, const int32_t* env_ids, int64_t n_ids, int64_t* episode_length,
             const AsResetOut* compact_out, void* stream) {
  AS_REQUIRE(h, "handle is null");
  const bool from_device_list = env_ids == nullptr && n_ids < 0;
  if (from_device_list) {
    // "the envs as_step_pass1 flagged": the id list that pass compacted on the device, however many there are
    if (!h->spec_valid) return fail(AS_ERR_STATE, "as_reset(env_ids = NULL, n_ids < 0) needs a preceding as_step_pass1");
    AS_REQUIRE(env_origins != nullptr, "env_origins is null");
  } else {
    AS_REQUIRE(n_ids >= 0 && n_ids <= h->num_envs, "id count out of range");
    if (n_ids == 0) return AS_OK;  // DRL:360: `_reset_idx` is not entered (an empty id tensor has a null pointer)
    AS_REQUIRE(env_origins && env_ids, "env_origins/env_ids is null");
  }
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  if (h->peer_three_call)
    if (int rc = check_peer(h)) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // (global 3-call mode: outside a step means "no pass 1 open" on every rank alike, whichever shard reset envs before)
  if (h->peer_three_call ? !h->spec_valid : !h->pass1_done) {
    // `_reset_idx` outside a step (DirectRLEnv.reset(), DRL:256-279): the promotion rule of ENV:471 looks at the
    // indices as they are now, and the draws must not repeat those of an earlier reset -- sum the indices and
    // advance the Philox step counter, which as_step_pass1 would have done
    k_prepare_reset<<<1, 1024, 0, s>>>(h->ws, h->num_envs);
    if (int rc = check_launch(h, "k_prepare_reset")) return rc;
    // global 3-call mode: the promotion on the global sum of the indices, pending grid outcomes into the histograms
    if (h->peer_three_call)
      if (int rc = launch_exchange(h, kExchangeReset, s)) return rc;
  }
  h->pass1_done = false;  // consumed: a second reset without a pass in between prepares for itself
  ResetArgs r = make_reset_args(h, env_origins);
  // (an explicit id list means `_reset_idx` was entered, i.e. some env reset; with the device-side list that is
  // decided by the count pass 1 folded -- the rule is not evaluated in a step in which nothing resets, DRL:360)
  r.force_any_reset = from_device_list ? 0 : 1;
  r.peer_decided = h->peer_three_call ? 1 : 0;
  if (compact_out) r.out = *compact_out;
  r.env_ids = from_device_list ? h->ws.reset_ids : env_ids;
  r.n_ids = from_device_list ? -1 : n_ids;
  h->device_list = from_device_list;
  r.ext_episode_length = episode_length;
  r.fused = 0;
  r.into_other = h->spec_valid ? 1 : 0;  // behind a speculating pass 1 the step continues in the other state buffer
  const bool regen_enabled = (h->params.flags & (AS_FLAG_GRID_CURRICULUM | AS_FLAG_INTENDED_REGEN)) != 0;
  // (k_reset_list lists the envs that regenerate: the list starts empty)
  if (regen_enabled) AS_CUDA(cudaMemsetAsync(&h->ws.ctrl->n_regen_list, 0, sizeof(uint32_t), s));
  // (four envs per warp; with the device-side list the count is only known on the device: sized for a tenth of the envs)
  const int grid = grid_for(from_device_list ? h->num_envs / 10 + 1 : n_ids, 32, h->sm_count, 3);
  k_reset_list<<<grid, 256, 0, s>>>(r);
  if (int rc = check_launch(h, "k_reset_list")) return rc;
  if (!regen_enabled) return AS_OK;
  // grid turnover and stones of the listed envs, by the kernel the fused step uses
  if (int rc = launch_regeneration(h, r, s)) return rc;
  // (k_pass2_commit clears the list when it closes the step; outside a step nothing follows that would, and a fused
  // step must start with an empty list)
  if (!r.into_other) AS_CUDA(cudaMemsetAsync(&h->ws.ctrl->n_regen_list, 0, sizeof(uint32_t), s));
  return AS_OK;
}

int as_step_pass2(AsHandle* h, const AsStateIn* in, float* obs, void* stream) {
  AS_REQUIRE(h && obs, "handle/obs is null");
  if (int rc = validate_state_in(h, in, false)) return rc;
  // (no call-order precondition: the reference runs `_compute_useful_values` at the end of `_reset_idx` whether or
  // not a pass preceded it -- DirectRLEnv.reset() calls `_reset_idx(all ids)` before the first step, DRL:256-279)
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  if (h->peer_three_call)
    if (int rc = check_peer(h)) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (h->spec_valid) {
    // pass 1 already ran pass 2 for every env that did not reset: redo the envs that did (from the views as they are
    // now, after the PhysX writes) and make the speculated state buffer the current one
    CommitArgs c;
    std::memset(&c, 0, sizeof(c));
    c.P = h->params;
    c.jc = h->jc;
    c.in = *in;
    c.ws = h->ws;
    c.obs = obs;
    c.obs_clip = h->obs_clip_pass1;
    c.inv_step_dt = h->inv_step_dt;
    c.num_envs = h->num_envs;
    c.revert_if_none = h->device_list ? 1 : 0;
    c.peer_three_call = h->peer_three_call ? 1 : 0;
    const int grid = grid_for(h->num_envs / 10 + 1, 32, h->sm_count, 3);
    k_pass2_commit<<<grid, 256, 0, s>>>(c);
    h->spec_valid = false;
    return check_launch(h, "k_pass2_commit");
  }
  AsStepOut out;
  std::memset(&out, 0, sizeof(out));
  out.obs = obs;
  out.obs_clip = h->obs_clip_pass1;
  StepArgs a = make_step_args(h, in, nullptr, 0, &out);
  const StepLaunch k = select_step(h, kModePass2, in, a);
  if (int rc = launch_prepare(h, in, s, a.body_from_prepare != 0)) return rc;
  AS_CUDA(launch_step(h, k, a, s));
  return check_launch(h, "k_step<pass2>");
}

int as_step_no_reset(AsHandle* h, void* stream) {
  AS_REQUIRE(h, "handle is null");
  if (!h->spec_valid) return AS_OK;  // nothing was speculated (no pass 1 since the last pass 2)
  if (h->peer_three_call)
    if (int rc = check_peer(h)) return rc;
  const int grid = grid_for(h->num_envs * 11, 256 * 4, h->sm_count, 8);
  k_pass2_revert<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(h->ws, h->spec_obs, h->obs_clip_pass1,
                                                                        h->num_envs, h->peer_three_call ? 1 : 0);
  h->spec_valid = false;
  return check_launch(h, "k_pass2_revert");
}

int as_apply_action(AsHandle* h, const float* actions, int64_t actions_stride, float* efforts, void* stream) {
  AS_REQUIRE(h && actions && efforts, "null argument");
  AS_REQUIRE(actions_stride >= kJ, "actions stride too small");
  // full tiles by TMA bulk copies: dense rows on 16-byte boundaries (a tile is 128 x 84 bytes)
  const bool bulk = actions_stride == kJ &&
                    ((reinterpret_cast<uintptr_t>(actions) | reinterpret_cast<uintptr_t>(efforts)) & 15u) == 0;
  const int tiles = bulk ? static_cast<int>(h->num_envs / kTile) : 0;
  const int64_t tail_items = (h->num_envs - static_cast<int64_t>(tiles) * kTile) * kJ;
  const int tail_blocks = tail_items ? grid_for(tail_items, 256 * 4, h->sm_count, 8) : 0;
  const int tile_blocks = (tiles + kActionTilesPerCta - 1) / kActionTilesPerCta;
  k_apply_action<<<tile_blocks + tail_blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      h->params, h->ws, actions, actions_stride, efforts, h->num_envs, tiles, tile_blocks, tail_blocks);
  return check_launch(h, "k_apply_action");
}

int as_mirror_batch(AsHandle* h, const AsMirrorJob* jobs, int32_t n_jobs, void* stream) {
  AS_REQUIRE(h && jobs, "null argument");
  AS_REQUIRE(n_jobs >= 1 && n_jobs <= 4, "1..4 jobs per launch");
  MirrorJobs mj;
  std::memset(&mj, 0, sizeof(mj));
  int64_t most_tiles = 0, most_tail = 0;
  for (int i = 0; i < n_jobs; ++i) {
    AS_REQUIRE(jobs[i].in && jobs[i].out, "job with a null pointer");
    AS_REQUIRE(jobs[i].rows >= 0, "negative row count");
    AS_REQUIRE(jobs[i].kind == 0 || jobs[i].kind == 1, "kind must be 0 (observations) or 1 (actions / mus)");
    const int64_t dim = jobs[i].kind == 0 ? kObs : kJ;
    AS_REQUIRE(jobs[i].rows * dim < (1ll << 40), "too many rows");
    mj.in[i] = jobs[i].in;
    mj.out[i] = jobs[i].out;
    mj.rows[i] = jobs[i].rows;
    mj.kind[i] = jobs[i].kind;
    // full tiles go through shared memory by TMA bulk copies: both halves of the output and the input on 16-byte
    // boundaries (torch allocations are; a row count that is a multiple of 4 puts the lower half on one too)
    const bool aligned = ((reinterpret_cast<uintptr_t>(jobs[i].in) | reinterpret_cast<uintptr_t>(jobs[i].out)) & 15u) == 0 &&
                         ((jobs[i].rows * dim * 4) & 15) == 0;
    const int64_t tiles = aligned ? jobs[i].rows / kMirrorRows : 0;
    AS_REQUIRE(tiles < (1ll << 30), "too many rows");
    mj.tiles[i] = static_cast<int32_t>(tiles);
    const int64_t tail_items = (jobs[i].rows - tiles * kMirrorRows) * dim;
    most_tiles = tiles > most_tiles ? tiles : most_tiles;
    most_tail = tail_items > most_tail ? tail_items : most_tail;
  }
  mj.n = n_jobs;
  if (most_tiles == 0 && most_tail == 0) return AS_OK;
  const int tail_blocks = most_tail ? grid_for(most_tail, 256 * 4, h->sm_count, 8) : 0;
  const dim3 grid(static_cast<unsigned>(most_tiles + tail_blocks), static_cast<unsigned>(n_jobs));
  k_mirror_batch<<<grid, 256, kMirrorSmemBytes, static_cast<cudaStream_t>(stream)>>>(h->mirror_obs, h->mirror_act, mj,
                                                                                     tail_blocks);
  return check_launch(h, "k_mirror_batch");
}

int as_mirror_rows(AsHandle* h, const float* in, float* out, int64_t rows, int32_t kind, void* stream) {
  AS_REQUIRE(h && in && out, "null argument");
  AS_REQUIRE(rows >= 0, "negative row count");
  AS_REQUIRE(kind == 0 || kind == 1, "kind must be 0 (observations) or 1 (actions)");
  if (rows == 0) return AS_OK;
  AsMirrorJob job;
  std::memset(&job, 0, sizeof(job));
  job.in = in;
  job.out = out;
  job.rows = rows;
  job.kind = kind;
  return as_mirror_batch(h, &job, 1, stream);
}

int as_export_state(AsHandle* h, const AsMdpState* dst, void* stream) {
  AS_REQUIRE(h && dst, "null argument");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  const int grid = grid_for(h->num_envs, 256, h->sm_count, 8);
  k_export<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(h->params, h->ws, *dst, h->num_envs);
  return check_launch(h, "k_export");
}

int as_export_stone_poses(AsHandle* h, const int32_t* env_ids, int64_t n_ids, float* view_poses, int32_t* view_ids,
                          void* stream) {
  AS_REQUIRE(h && view_poses, "null argument");
  AS_REQUIRE(n_ids >= 0 && n_ids <= h->num_envs, "n_ids out of range");
  const int S = handle_stones(h);
  AS_REQUIRE(h->num_envs * S < (1ll << 31), "view indices must fit 32 bits");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  if (!env_ids) n_ids = h->num_envs;
  if (n_ids == 0) return AS_OK;
  const int grid = grid_for(n_ids * S, 256, h->sm_count, 8);
  k_export_stone_poses<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(h->ws, env_ids, n_ids, h->num_envs, S,
                                                                             view_poses, view_ids);
  return check_launch(h, "k_export_stone_poses");
}

int as_import_state(AsHandle* h, const AsMdpState* src, void* stream) {
  AS_REQUIRE(h && src, "null argument");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(h->num_envs, 256, h->sm_count, 8);
  k_import<<<grid, 256, 0, s>>>(h->params, h->ws, *src, h->num_envs);
  if (int rc = check_launch(h, "k_import")) return rc;
  k_clear_promotion<<<1, 32, 0, s>>>(h->ws.ctrl);
  return check_launch(h, "k_clear_promotion");
}

// Snapshot layout: [Ctrl | state words, both buffers | stone windows | grid bins | window-stale bits | stones (optional)].
namespace {
struct SnapshotLayout {
  int64_t ctrl, state, window, bin, stale, stones, total;
};
SnapshotLayout snapshot_layout(int64_t n, int S, bool with_stones) {
  const WorkspaceLayout w = workspace_layout(n, S);
  SnapshotLayout l;
  int64_t off = 0;
  l.ctrl = off;   off += w.state0_off - w.ctrl_off;
  l.state = off;  off += w.stones_off - w.state0_off;
  l.window = off; off += w.reset_ids_off - w.window_off;
  l.bin = off;    off += w.contact_pre_off - w.bin_off;
  l.stale = off;  off += w.total - w.win_stale_off;
  l.stones = off; off += with_stones ? (w.window_off - w.stones_off) : 0;
  l.total = off;
  return l;
}
}  // namespace

int64_t as_snapshot_bytes(const AsHandle* h, int32_t include_stones) {
  if (!h) return 0;
  return snapshot_layout(h->num_envs, handle_stones(h), include_stones != 0).total;
}

int as_snapshot(AsHandle* h, void* dst, int32_t include_stones, void* stream) {
  AS_REQUIRE(h && dst, "null argument");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const WorkspaceLayout w = workspace_layout(h->num_envs, handle_stones(h));
  const SnapshotLayout l = snapshot_layout(h->num_envs, handle_stones(h), include_stones != 0);
  unsigned char* d = static_cast<unsigned char*>(dst);
  const unsigned char* base = reinterpret_cast<const unsigned char*>(h->ws.ctrl);
  AS_CUDA(cudaMemcpyAsync(d + l.ctrl, base + w.ctrl_off, static_cast<size_t>(l.window - l.ctrl), cudaMemcpyDeviceToDevice, s));
  AS_CUDA(cudaMemcpyAsync(d + l.window, base + w.window_off, static_cast<size_t>(l.bin - l.window), cudaMemcpyDeviceToDevice, s));
  AS_CUDA(cudaMemcpyAsync(d + l.bin, base + w.bin_off, static_cast<size_t>(l.stale - l.bin), cudaMemcpyDeviceToDevice, s));
  AS_CUDA(cudaMemcpyAsync(d + l.stale, base + w.win_stale_off, static_cast<size_t>(l.stones - l.stale), cudaMemcpyDeviceToDevice, s));
  if (include_stones)
    AS_CUDA(cudaMemcpyAsync(d + l.stones, base + w.stones_off, static_cast<size_t>(l.total - l.stones), cudaMemcpyDeviceToDevice, s));
  return AS_OK;
}

int as_restore(AsHandle* h, const void* src, int32_t include_stones, void* stream) {
  AS_REQUIRE(h && src, "null argument");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const WorkspaceLayout w = workspace_layout(h->num_envs, handle_stones(h));
  const SnapshotLayout l = snapshot_layout(h->num_envs, handle_stones(h), include_stones != 0);
  const unsigned char* d = static_cast<const unsigned char*>(src);
  unsigned char* base = reinterpret_cast<unsigned char*>(h->ws.ctrl);
  k_restore_ctrl<<<1, 256, 0, s>>>(h->ws.ctrl, reinterpret_cast<const Ctrl*>(d + l.ctrl));
  if (int rc = check_launch(h, "k_restore_ctrl")) return rc;
  AS_CUDA(cudaMemcpyAsync(base + w.state0_off, d + l.state, static_cast<size_t>(l.window - l.state), cudaMemcpyDeviceToDevice, s));
  AS_CUDA(cudaMemcpyAsync(base + w.window_off, d + l.window, static_cast<size_t>(l.bin - l.window), cudaMemcpyDeviceToDevice, s));
  AS_CUDA(cudaMemcpyAsync(base + w.bin_off, d + l.bin, static_cast<size_t>(l.stale - l.bin), cudaMemcpyDeviceToDevice, s));
  AS_CUDA(cudaMemcpyAsync(base + w.win_stale_off, d + l.stale, static_cast<size_t>(l.stones - l.stale), cudaMemcpyDeviceToDevice, s));
  if (include_stones)
    AS_CUDA(cudaMemcpyAsync(base + w.stones_off, d + l.stones, static_cast<size_t>(l.total - l.stones), cudaMemcpyDeviceToDevice, s));
  h->pass1_done = false;
  return AS_OK;
}

int as_grid_state(AsHandle* h, uint8_t* bins_dst, const uint8_t* bins_src, uint32_t* hist_dst, const uint32_t* hist_src,
                  void* stream) {
  AS_REQUIRE(h, "handle is null");
  if (h->pending_valid) return fail(AS_ERR_STATE, "a fused step is open; close it with as_finish_step");
  const int grid = grid_for(h->num_envs > kMaxGridBins ? h->num_envs : kMaxGridBins, 256, h->sm_count, 8);
  k_grid_state<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(h->ws, bins_dst, bins_src, hist_dst, hist_src,
                                                                     h->num_envs);
  return check_launch(h, "k_grid_state");
}

int as_set_timing_events(AsHandle* h, void* start_event, void* stop_event) {
  AS_REQUIRE(h, "handle is null");
  AS_REQUIRE((start_event == nullptr) == (stop_event == nullptr), "give both events or none");
  h->ev_start = static_cast<cudaEvent_t>(start_event);
  h->ev_stop = static_cast<cudaEvent_t>(stop_event);
  return AS_OK;
}

int as_debug_timing(AsHandle* h, uint64_t* host16, int reset, void* stream) {
  AS_REQUIRE(h && host16, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  AS_CUDA(cudaMemcpyAsync(host16, h->ws.ctrl->dbg_t, 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  if (reset) AS_CUDA(cudaMemsetAsync(h->ws.ctrl->dbg_t, 0, 16 * sizeof(uint64_t), s));
  AS_CUDA(cudaStreamSynchronize(s));
  return AS_OK;
}

int64_t as_launch_count(const AsHandle* h) { return h ? h->launches : 0; }

int64_t as_sizeof(int32_t which) {
  switch (which) {
    case 0: return sizeof(AsParams);
    case 1: return sizeof(AsStateIn);
    case 2: return sizeof(AsStepOut);
    case 3: return sizeof(AsResetOut);
    case 4: return sizeof(AsStats);
    case 5: return sizeof(AsMdpState);
    case 6: return sizeof(AsMirrorJob);
    case 7: return sizeof(AsExchange);
    default: return -1;
  }
}

int as_stats_device_ptr(AsHandle* h, AsStats** device_stats) {
  AS_REQUIRE(h && device_stats, "null argument");
  *device_stats = &h->ws.ctrl->stats;
  return AS_OK;
}

int as_read_stats(AsHandle* h, AsStats* host_out, void* stream) {
  AS_REQUIRE(h && host_out, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  AS_CUDA(cudaMemcpyAsync(host_out, &h->ws.ctrl->stats, sizeof(AsStats), cudaMemcpyDeviceToHost, s));
  AS_CUDA(cudaStreamSynchronize(s));
  return AS_OK;
}

}  // extern "C"
