// rd_env.cu -- librd_env.so: the C ABI of include/rd_env.h over the sm_100a kernels.
//
// One handle = one CUDA device, one batch of envs.  The library owns the env state (SoA float64/int32),
// the uploaded maps and a few scratch arrays; every I/O buffer is a caller-owned device pointer.
// There is no CPU path: rd_create fails with RD_ERR_NO_DEVICE when no sm_100 device is usable.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "rd_common.cuh"
#include "rd_dynamics.cuh"
#include "rd_lidar.cuh"
#include "rd_occupancy.cuh"
#include "rd_policy.cuh"
#include "rd_dreamer.cuh"
#include "rd_store.cuh"

#define RD_API extern "C" __attribute__((visibility("default")))

namespace {

thread_local std::string g_last_error;

struct HostMap {
  DevMap dev{};
  void* d_bits = nullptr;
  void* d_dist = nullptr;
  void* d_start = nullptr;
  void* d_reset = nullptr;
  void* d_next = nullptr;
  size_t hot_bytes = 0;    // bytes of the d_bits allocation (bits + clearance + distance): the L2-persisting window
  bool present = false;
  int lidar_per_sm[12] = {-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1};   // resident k_lidar CTAs per SM for this map, per kernel
                                                            // instantiation (cached launch configuration)
};

}  // namespace

struct rd_env {
  rd_config cfg{};
  int device = 0;
  int sm_count = 0;
  int smem_optin = 0;             // max dynamic shared memory per CTA (opt-in), bytes
  int smem_per_sm = 0;            // shared memory per SM, bytes
  size_t l2_window_max = 0;       // > 0: L2 persistence is set up; the largest access-policy window the device takes
  bool lidar_centre_first = true; // k_lidar work order (RD_LIDAR_ORDER=0: env-major)
  bool lidar_attr_set[12] = {};   // k_lidar<16|24|32, groups per item, cars> opted in to smem_optin
  int n = 0;
  int step_block = 128;           // k_step threads per CTA (small batches: fewer, so that every SM gets a warp)
  bool step_split = true;         // k_step_split (two warps per 32 envs) while the batch is latency-bound; RD_STEP_SPLIT overrides
  double2* d_f2 = nullptr;        // env state, SoA of 16-byte groups (rd_dynamics.cuh StateRef)
  int4* d_i4 = nullptr;
  int2* d_i2 = nullptr;
  VehConst vk{};                  // vehicle constants of cfg.vehicle / cfg.dt (rd_vehicle.cuh)
  VehAcc voff{};
  VehConst* d_vk = nullptr;       // device copies of the two (rdv_tick's out-of-line general path reads them through pointers)
  VehAcc* d_voff = nullptr;
  double* d_stats = nullptr;
  double* d_hist = nullptr;       // [n_step_progress][n] ring of lap + progress (n_step_progress task), else null
  bool multi = false;             // k_step_ma steps the batch (agents_per_world > 1 or an n_step_progress task)
  OriginRec* d_recs = nullptr;
  double* d_beam_tab = nullptr;
  DevMap* d_maps = nullptr;
  int32_t* d_env_order = nullptr;  // env indices grouped by map
  unsigned int* d_lidar_ctr = nullptr;  // [RD_CTR_RING][2] work counter + finish ticket of k_lidar (self re-arming); every
  unsigned lidar_ctr_next = 0;          // launch takes the next pair of the ring, so launches that overlap (programmatic
                                        // dependent launch, calls on different streams) never share a counter
  OccScratch occ{};
  HostMap maps[RD_MAX_MAPS];
  std::vector<int> order_offset;   // RD_MAX_MAPS + 1 offsets into d_env_order
  bool maps_dirty = true, assigned = false, was_reset = false;
  // scratch for the stage entry points
  OriginRec* d_stage_recs = nullptr;
  int32_t* d_stage_ids = nullptr;
  int stage_cap = 0;
  int64_t launches = 0;
  std::vector<int32_t> h_order;     // host copy of d_env_order (chunk -> per-map sub-ranges)
  // host-facing path (rd_host_init / rd_step_host)
  struct HostPath {
    bool ready = false;
    int n_chunks = 0;
    std::vector<int> bounds;                 // n_chunks + 1 env indices
    std::vector<cudaStream_t> streams;
    std::vector<cudaEvent_t> ev_done;
    cudaEvent_t ev_act = nullptr;
    float* act_host = nullptr; float* act_dev = nullptr;
    uint8_t* mask_dev = nullptr;
    unsigned char* small_dev = nullptr; unsigned char* small_host = nullptr; size_t small_bytes = 0;
    float* lidar_dev = nullptr; float* lidar_host = nullptr;   // float32 rows, or IEEE half rows (lidar_elem == 2)
    size_t lidar_elem = 4;
    uint8_t* occ_dev = nullptr; uint8_t* occ_host = nullptr;
    bool pending = false;                    // rd_step_host_begin enqueued a step whose results rd_step_host_end has not awaited
    rd_outputs dev_out{}, host_out{};
  } hp;
  // on-device follow-the-gap controller (rd_policy_gap_follower_init)
  struct Policy {
    bool ready = false;
    rd_gap_follower g{};
    PolicyState st{};
    float* d_actions = nullptr;   // [n][2] rollout scratch
    bool attr_set = false;        // kernel opted in to > 48 KB of dynamic shared memory
  } pol;
  DreamerPolicy dr;   // on-device Dreamer agent (rd_policy_dreamer_init)
  // device-resident episode store (rd_store_init, csrc/rd_store.cuh)
  struct Store {
    bool ready = false, started = false;   // started: rd_store_reset has run
    rd_store_config sc{};
    int64_t max_steps = 0;
    StoreDev d{};
    uint8_t* d_all = nullptr;               // [n] ones: the reset mask of rd_store_reset
    unsigned long long* d_invalid = nullptr;
    int64_t* d_elig = nullptr; int* d_n_elig = nullptr;   // eligibility compaction (ids in commit order, count)
    void* d_cub = nullptr; size_t cub_bytes = 0;
    int64_t epoch = 0, elig_epoch = -1; int elig_min = -1;   // the compaction is redone when the store or min_len changed
    int64_t* d_req_id = nullptr; int32_t* d_req_start = nullptr; int req_cap = 0;
    int64_t* d_export = nullptr;            // [M + Mi][3] (id, env, rows) of rd_store_info
    int64_t draws = 0;
    int32_t* d_imp_len = nullptr; int64_t* d_imp_first = nullptr; int imp_meta_cap = 0;   // rd_store_import: per episode
  } st;
  // device-resident steps over several tracks: the observation kernels of every track but the first run on their own
  // stream (fork behind the step kernel, join at the end), so that a track's kernels fill the SMs the previous track's
  // persistent CTAs leave in their tail.  RD_FORK_MAPS=0 keeps everything on the caller's stream.
  bool fork_maps = true;
  bool in_fork = false;           // set while observe() enqueues a forked track's kernels
  cudaStream_t map_stream[RD_MAX_MAPS] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[RD_MAX_MAPS] = {};
  // optional per-kernel timing (rd_enable_timing)
  bool timing = false;
  struct Timed { cudaEvent_t a, b; int kind; };
  std::vector<Timed> timed;
  std::vector<cudaEvent_t> event_pool;
  rd_timing acc{};
  std::string error;
};

namespace {

int fail(rd_env* env, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  if (env) env->error = buf;
  return code;
}

#define CUDA_TRY(env, expr)                                                                         \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      cudaGetLastError(); /* do not leave the error sticky for the caller's own CUDA calls */       \
      return fail(env, RD_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e));                       \
    }                                                                                               \
  } while (0)

void default_config(rd_config* c) {
  std::memset(c, 0, sizeof(*c));
  c->abi_version = RD_ABI_VERSION;
  c->n_envs = 1;
  c->n_beams = 1080;          // [REF dreamer/dream.py:66]
  c->action_repeat = 4;       // [REF dreamer/dream.py:55]
  c->repeat_semantics = RD_REPEAT_DREAMER;
  c->obs_flags = RD_OBS_LIDAR;
  c->task = RD_TASK_MAX_PROGRESS;
  c->laps = 10;               // [REF dreamer/scenarios/max_progress/austria.yml:10]
  c->terminate_on_collision = 1;
  c->n_checkpoints = 20;
  c->time_limit_steps = 0;
  c->auto_reset = 0;
  c->reset_mode = RD_RESET_GRID;
  c->rescale_actions = 1;
  c->clip_actions = 0;
  c->progress_abs = 0;
  c->env_id_offset = 0;
  c->seed = 0;
  c->dt = 0.01;               // [REF dreamer/callbacks.py:23]
  c->time_limit = 180.0;
  c->collision_reward = -1.0;
  c->progress_reward = 100.0;
  c->frame_reward = 0.0;
  c->action_low[0] = 0.005; c->action_low[1] = -1.0;   // [REF dreamer/dream.py:138]
  c->action_high[0] = 1.0;  c->action_high[1] = 1.0;
  c->lidar_fov = 270.0 * (3.14159265358979323846 / 180.0);  // [REF dreamer/tools.py:84-86]
  c->lidar_range_min = 0.25;
  c->lidar_range_max = 15.0;  // [REF dreamer/tools.py:274]
  c->lidar_offset = 0.0;
  c->lidar_noise = 0.0f;
  c->agents_per_world = 1;
  for (int a = 0; a < RD_MAX_AGENTS; ++a) c->agent_task[a] = RD_TASK_MAX_PROGRESS;
  c->n_step_progress = 10;    // [REF baselines/scenarios/max_progress/austria.yml:18]
  c->ball_spacing = 1.5;
  c->time_limit_ticks = 0;
  // Box bounds of the env's observation space [NEW-SPEC: racecar_gym's sensor spaces are not in tree]: lidar [0, range],
  // pose +-100 m (the maps span +-50 m), velocity +-10 (v_max = 5 m/s)
  c->obs_low[RD_NORM_LIDAR] = 0.0;      c->obs_high[RD_NORM_LIDAR] = 15.0;
  c->obs_low[RD_NORM_POSE] = -100.0;    c->obs_high[RD_NORM_POSE] = 100.0;
  c->obs_low[RD_NORM_VELOCITY] = -10.0; c->obs_high[RD_NORM_VELOCITY] = 10.0;
  rd_vehicle* v = &c->vehicle;
  v->mu = 1.0489; v->c_sf = 4.718; v->c_sr = 5.4562; v->lf = 0.15875; v->lr = 0.17145; v->h_cg = 0.074;
  v->mass = 3.74; v->inertia = 0.04712;
  v->steer_min = -0.42; v->steer_max = 0.42; v->steer_vel_max = 3.2;  // [REF ros_agent/models/dreamer/racing_dreamer.py:14]
  v->v_switch = 7.319; v->a_max = 9.51; v->v_min = 0.0; v->v_max = 5.0;  // [REF racing_dreamer.py:16]
  v->v_kinematic = 0.5;
  v->a_drive = 6.0; v->a_brake = 8.26; v->c_drag = 1.0;  // [REF ros_agent/agents/follow_the_gap/src/agent.py:74]
  // sign: a positive steering action turns RIGHT, as in the reference's simulator (racecar_gym drives the steering joint to
  // -steering * max_angle); in-tree evidence: the ROS node negates the agent's steering for the left-positive Ackermann
  // message [REF ros_agent/agents/dreamer/src/agent.py:111], and the shipped Dreamer agents only drive with this sign.
  v->steer_gain = -1.0;
  v->body_length = 0.50; v->body_width = 0.27;
}

// k_lidar work-counter pairs: far more than the launches one handle can have in flight (the host-facing step enqueues at
// most chunks x maps <= 24 x 8 launches before it waits)
constexpr int RD_CTR_RING = 1024;

int sync_maps(rd_env* env) {
  if (!env->maps_dirty) return RD_OK;
  DevMap host[RD_MAX_MAPS];
  for (int i = 0; i < RD_MAX_MAPS; ++i) host[i] = env->maps[i].dev;
  CUDA_TRY(env, cudaMemcpy(env->d_maps, host, sizeof(host), cudaMemcpyHostToDevice));
  env->maps_dirty = false;
  return RD_OK;
}

enum { T_STEP = 0, T_LIDAR = 1, T_OCC = 2, T_RESET = 3, T_POLICY = 4 };

cudaEvent_t take_event(rd_env* env) {
  if (!env->event_pool.empty()) { cudaEvent_t e = env->event_pool.back(); env->event_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
// brackets the launches issued during its lifetime with two events on `s`
struct ScopedTiming {
  rd_env* env; cudaStream_t s; int kind; cudaEvent_t a = nullptr;
  ScopedTiming(rd_env* e, cudaStream_t st, int k, bool on = true) : env(e), s(st), kind(k) {
    if (env->timing && on) { a = take_event(env); cudaEventRecord(a, s); }
  }
  ~ScopedTiming() {
    if (a) { cudaEvent_t b = take_event(env); cudaEventRecord(b, s); env->timed.push_back({a, b, kind}); }
  }
};

LidarParams lidar_params(const rd_env* env, const DevMap& m) {
  const rd_config& c = env->cfg;
  LidarParams lp{};
  lp.n_beams = c.n_beams;
  lp.groups = (c.n_beams + 31) / 32;
  lp.gpi = 1;
  lp.units = lp.groups;
  lp.groups_magic = lp.units > 1 ? (unsigned)(((1ull << 32) + (unsigned)lp.units - 1) / (unsigned)lp.units) : 0u;
  lp.normalize = (c.obs_flags & RD_OBS_LIDAR_NORM) ? 1 : ((c.obs_flags & RD_OBS_NORM_BASELINES) ? 2 : 0);
  lp.norm_lo = c.obs_low[RD_NORM_LIDAR];
  lp.norm_sc = 1.0 / (c.obs_high[RD_NORM_LIDAR] - c.obs_low[RD_NORM_LIDAR]);
  lp.f16 = (c.obs_flags & RD_OBS_LIDAR_F16) ? 1 : 0;
  lp.range_min = (float)c.lidar_range_min;
  lp.range_max = (float)c.lidar_range_max;
  lp.noise = c.lidar_noise;
  lp.scale = (float)((double)(1 << (RD_DIR_BITS - RD_SUB_BITS)) * m.res);
  lp.rsub = (int64_t)std::rint(c.lidar_range_max * m.inv_res * (double)RD_SUB);
  lp.key0 = (uint32_t)c.seed;
  lp.key1 = (uint32_t)(c.seed >> 32) ^ RD_STREAM_LIDAR;
  lp.agents = c.agents_per_world > 1 ? c.agents_per_world : 1;
  {  // body box of another car in ITS sensor frame (the record holds the sensor origin), in cells, as float32
    const double hl = 0.5 * c.vehicle.body_length * m.inv_res, hw = 0.5 * c.vehicle.body_width * m.inv_res;
    const double off = c.lidar_offset * m.inv_res;
    lp.car_ulo = (float)(-hl - off);
    lp.car_uhi = (float)(hl - off);
    lp.car_hw = (float)hw;
    lp.res = (float)m.res;
    lp.car_radius_sub = (int)std::ceil((hl + hw + std::fabs(off) + 1.0) * (double)RD_SUB);
    lp.car_reach = (int)std::ceil((c.lidar_range_max * m.inv_res + 2.0 * (hl + hw + std::fabs(off)) + 2.0) * (double)RD_SUB);
  }
  return lp;
}

// Launch attributes shared by the step and LiDAR kernels: (optionally) programmatic dependent launch, and an L2
// access-policy window that marks the track's hot arrays (bit grid, clearance field, wavefront distance: 0.1-1.3 MB)
// as PERSISTING, so that whatever runs between two env steps (a learner's GEMMs, bench.py's 256 MB flush) does not evict
// the map [north_star: "L2 residency control on the map"].  rd_create sets aside the persisting share of L2 once.
int launch_attrs(const rd_env* env, int map_id, bool pdl, cudaLaunchAttribute* at) {
  int n = 0;
  if (pdl) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (env->l2_window_max > 0 && map_id >= 0 && env->maps[map_id].present && env->maps[map_id].hot_bytes > 0) {
    const HostMap& m = env->maps[map_id];
    at[n].id = cudaLaunchAttributeAccessPolicyWindow;
    at[n].val.accessPolicyWindow.base_ptr = m.d_bits;
    at[n].val.accessPolicyWindow.num_bytes = std::min(m.hot_bytes, env->l2_window_max);
    at[n].val.accessPolicyWindow.hitRatio = 1.0f;
    at[n].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    at[n].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    ++n;
  }
  return n;
}

// LiDAR launch for the envs of one map: persistent CTAs, grid = resident CTAs on all SMs.
template <int WARPS, int GPI, bool CARS>
int launch_lidar_t(rd_env* env, int map_id, const OriginRec* recs, const int32_t* order, int n_env, float* out,
                   cudaStream_t s, unsigned int* ctr) {
  const DevMap& m = env->maps[map_id].dev;
  LidarParams lp = lidar_params(env, m);
  lp.centre_first = env->lidar_centre_first ? 1 : 0;
  lp.envs_magic = n_env > 1 ? (unsigned)(((1ull << 32) + (unsigned)n_env - 1) / (unsigned)n_env) : 0u;
  const size_t tab_bytes = ((size_t)2 * lp.n_beams * 8 + 15) & ~(size_t)15;
  const size_t smem = 16 + tab_bytes + (size_t)m.bits_bytes;
  auto kern = k_lidar<WARPS, GPI, CARS>;
  // which instantiation runs depends on the map (warps), the handle (cars) AND the launch size (groups per item), so both
  // the opt-in to the device's shared-memory maximum and the cached occupancy are kept per instantiation
  const int variant = (WARPS == 32 ? 2 : (WARPS == 24 ? 1 : 0)) + (GPI == 2 ? 3 : 0) + (CARS ? 6 : 0);
  bool& attr = env->lidar_attr_set[variant];
  if (!attr) {
    CUDA_TRY(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, env->smem_optin));
    attr = true;
  }
  int& per_sm = env->maps[map_id].lidar_per_sm[variant];
  if (per_sm < 0) {  // once per map and instantiation: ask how many CTAs fit on an SM
    if (smem > (size_t)env->smem_optin) return fail(env, RD_ERR_INVALID, "map %d (%zu B) does not fit in shared memory", map_id, smem);
    int q = 0;
    CUDA_TRY(env, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, WARPS * 32, smem));
    if (q < 1) return fail(env, RD_ERR_INVALID, "map %d (%zu B) does not fit in shared memory", map_id, smem);
    per_sm = q;
  }
  lp.gpi = GPI;
  lp.units = (lp.groups + GPI - 1) / GPI;
  lp.groups_magic = lp.units > 1 ? (unsigned)(((1ull << 32) + (unsigned)lp.units - 1) / (unsigned)lp.units) : 0u;
  const long long items = (long long)n_env * lp.units;
  if (items >= (1ll << 31)) return fail(env, RD_ERR_INVALID, "too many (env, beam group) items for one launch");
  // rd_march keeps the ray position in 32-bit 2^-18 cells (rd_march.cuh)
  if ((long long)std::max(m.w, m.h) + (lp.rsub >> RD_SUB_BITS) >= 8190)
    return fail(env, RD_ERR_INVALID, "map %d (%d x %d cells) plus the LiDAR range (%lld cells) exceeds the ray march's 8190-cell span",
                map_id, m.w, m.h, (long long)(lp.rsub >> RD_SUB_BITS));
  long long grid = std::min<long long>((items + WARPS - 1) / WARPS, (long long)env->sm_count * per_sm);
  if (grid < 1) return RD_OK;
  {
    // (a forked track's launch queues behind the first track's persistent CTAs: its event bracket would measure the
    // wait, so only launches on the caller's stream are timed)
    ScopedTiming tm(env, s, T_LIDAR, !env->in_fork);
    // Programmatic dependent launch: k_lidar's set-up (mbarrier, the bulk copy of the map into shared memory, the beam
    // table, the first draw from the work counter) overlaps the tail of the kernel in front of it on the stream
    // (k_step / k_reset trigger early with griddepcontrol.launch_dependents); k_lidar executes griddepcontrol.wait before
    // it touches the origin records.
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(WARPS * 32); lc.dynamicSmemBytes = smem; lc.stream = s;
    cudaLaunchAttribute at[2];
    lc.attrs = at; lc.numAttrs = launch_attrs(env, map_id, true, at);
    const DevMap* a_maps = env->d_maps; const double* a_tab = env->d_beam_tab;
    cudaError_t le = cudaLaunchKernelEx(&lc, kern, a_maps, map_id, recs, order, n_env, lp, a_tab, out, ctr);
    if (le != cudaSuccess) { cudaGetLastError(); return fail(env, RD_ERR_CUDA, "k_lidar launch: %s", cudaGetErrorString(le)); }
  }
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}

int launch_lidar(rd_env* env, int map_id, const OriginRec* recs, const int32_t* order, int n_env, float* out,
                 cudaStream_t s, unsigned int* ctr = nullptr) {
  const DevMap& m = env->maps[map_id].dev;
  if (!ctr) ctr = env->d_lidar_ctr + 2 * (env->lidar_ctr_next++ % RD_CTR_RING);
  // 48 resident warps per SM wherever the shared-memory copies of the map allow it (the kernel is capped at 40
  // registers for that): three 16-warp CTAs for small maps, two 24-warp CTAs for maps of which two copies fit, one
  // 32-warp CTA otherwise.
  const size_t smem1 = 16 + (((size_t)2 * env->cfg.n_beams * 8 + 15) & ~(size_t)15) + (size_t)m.bits_bytes + 1024;   // + the per-CTA reserve
  const size_t sm_total = (size_t)env->smem_per_sm;
  const int warps = 3 * smem1 <= sm_total ? 16 : (2 * smem1 <= sm_total ? 24 : 32);
  // Two beam groups per work item once a resident warp gets enough of them (see k_lidar): 45 groups per warp is where
  // the curves cross (profiles/r3o_lidar_groups_per_item.txt).
  const long long resident_warps = (long long)env->sm_count * (warps == 32 ? 32 : 48);
  const int gpi = (long long)n_env * ((env->cfg.n_beams + 31) / 32) >= 45LL * resident_warps ? 2 : 1;
  const bool cars = env->cfg.agents_per_world > 1;   // worlds: the scans also see the other cars (own instantiation, so
                                                      // that the single-car kernel keeps its register budget)
#define RD_LIDAR_GO(W, G, C) launch_lidar_t<W, G, C>(env, map_id, recs, order, n_env, out, s, ctr)
#define RD_LIDAR_GO_W(W) (cars ? (gpi == 2 ? RD_LIDAR_GO(W, 2, true) : RD_LIDAR_GO(W, 1, true)) \
                               : (gpi == 2 ? RD_LIDAR_GO(W, 2, false) : RD_LIDAR_GO(W, 1, false)))
  if (warps == 32) return RD_LIDAR_GO_W(32);
  if (warps == 24) return RD_LIDAR_GO_W(24);
  return RD_LIDAR_GO_W(16);
#undef RD_LIDAR_GO_W
#undef RD_LIDAR_GO
}

int launch_occupancy(rd_env* env, int map_id, const OriginRec* recs, const double* poses_xyyaw,
                     const int32_t* order, int n_env, uint8_t* out, cudaStream_t s) {
  ScopedTiming tm(env, s, T_OCC, !env->in_fork);
  int rc = occ_launch(env->occ, env->d_maps, map_id, env->maps[map_id].dev, recs, poses_xyyaw, env->d_f2, env->n,
                      order, n_env, out, env->sm_count, s, &env->launches);
  if (rc != 0) return fail(env, RD_ERR_CUDA, "occupancy launch: %s", cudaGetErrorString((cudaError_t)rc));
  return RD_OK;
}

OutPtrs out_ptrs(const rd_outputs* o) {
  OutPtrs p{};
  if (o) {
    p.pose = o->pose_dev; p.velocity = o->velocity_dev; p.speed = o->speed_dev; p.reward = o->reward_dev;
    p.done = o->done_dev; p.progress = o->progress_dev; p.lap = o->lap_dev; p.time = o->time_dev;
    p.flags = o->flags_dev; p.occupancy = o->occupancy_dev; p.rank = o->rank_dev; p.opponents = o->opponents_dev;
    p.wrong_way = o->wrong_way_dev; p.wall_collision = o->wall_collision_dev;
  }
  return p;
}

StepParams step_params(rd_env* env) {
  StepParams P{};
  P.cfg = env->cfg;
  P.vk = env->vk; P.off = env->voff; P.vk_g = env->d_vk; P.off_g = env->d_voff;
  P.S.f2 = env->d_f2; P.S.i4 = env->d_i4; P.S.i2 = env->d_i2; P.S.n = env->n;
  P.stats = env->d_stats; P.recs = env->d_recs; P.maps = env->d_maps;
  P.norm = (env->cfg.obs_flags & RD_OBS_NORM_BASELINES) ? 1 : 0;
  for (int k = 0; k < 3; ++k) {
    P.norm_lo[k] = env->cfg.obs_low[k];
    P.norm_sc[k] = P.norm ? 1.0 / (env->cfg.obs_high[k] - env->cfg.obs_low[k]) : 1.0;
  }
  P.pol = env->pol.st;
  P.hist = env->d_hist;
  if (env->dr.ready) { P.pol.dr_feat = env->dr.feat[env->dr.cur].p[0]; P.pol.dr_feat_lo = env->dr.feat[env->dr.cur].p[1]; P.pol.dr_ld = env->dr.ldf; P.pol.dr_row = env->dr.row_of_env; }
  P.n = env->n;
  return P;
}

// the dynamics / reward / termination kernel over the whole batch: k_step (independent cars) or k_step_ma (worlds)
int launch_step(rd_env* env, const rd_outputs* out, const float* actions_dev, cudaStream_t s) {
  {
    ScopedTiming tm(env, s, T_STEP);
    // the L2 window of the step kernel covers the track most envs drive on (one window per launch)
    int hot = -1, most = 0;
    for (int mid = 0; mid < RD_MAX_MAPS; ++mid) {
      const int cnt = env->order_offset[mid + 1] - env->order_offset[mid];
      if (cnt > most) { most = cnt; hot = mid; }
    }
    cudaLaunchAttribute at[2];
    cudaLaunchConfig_t lc{};
    lc.stream = s; lc.attrs = at; lc.numAttrs = launch_attrs(env, hot, false, at);
    const int tb = env->step_block;
    const StepParams P = step_params(env);
    const OutPtrs o = out_ptrs(out);
    cudaError_t le;
    if (env->multi) {
      const int A = env->cfg.agents_per_world > 1 ? env->cfg.agents_per_world : 1;
      const int per_cta = (tb / A) * A;
      lc.gridDim = dim3((unsigned)((env->n + per_cta - 1) / per_cta)); lc.blockDim = dim3(tb);
      le = cudaLaunchKernelEx(&lc, k_step_ma, P, o, actions_dev);
    } else if (env->step_split && env->cfg.action_repeat <= RD_SPLIT_TICKS) {
      // five warps per 32 envs (dynamics | position | probe | bookkeeping | reset look-ahead): shortens the per-env
      // latency chain k_step is bound by
      lc.gridDim = dim3((unsigned)((env->n + 31) / 32)); lc.blockDim = dim3(160);
      le = cudaLaunchKernelEx(&lc, k_step_split, P, o, actions_dev, 0, env->n);
    } else {
      lc.gridDim = dim3((unsigned)((env->n + tb - 1) / tb)); lc.blockDim = dim3(tb);
      le = cudaLaunchKernelEx(&lc, k_step, P, o, actions_dev, 0, env->n);
    }
    if (le != cudaSuccess) { cudaGetLastError(); return fail(env, RD_ERR_CUDA, "k_step launch: %s", cudaGetErrorString(le)); }
  }
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}

// LiDAR / occupancy launches for the envs [e0, e1) (grouped by map; each map's env list is ascending)
int observe(rd_env* env, const rd_outputs* out, cudaStream_t s, int e0 = 0, int e1 = -1, unsigned int* ctr = nullptr,
            bool fork = false) {
  if (!out) return RD_OK;
  if (e1 < 0) e1 = env->n;
  int tracks = 0;
  for (int mid = 0; mid < RD_MAX_MAPS; ++mid) tracks += env->order_offset[mid + 1] > env->order_offset[mid] ? 1 : 0;
  fork = fork && env->fork_maps && tracks > 1;
  bool forked[RD_MAX_MAPS] = {};
  int seen = 0;
  for (int mid = 0; mid < RD_MAX_MAPS; ++mid) {
    const int32_t* hb = env->h_order.data() + env->order_offset[mid];
    const int32_t* he = env->h_order.data() + env->order_offset[mid + 1];
    const int first = (int)(std::lower_bound(hb, he, e0) - hb), last = (int)(std::lower_bound(hb, he, e1) - hb);
    const int n_env = last - first;
    if (n_env == 0) continue;
    const int32_t* order = env->d_env_order + env->order_offset[mid] + first;
    cudaStream_t sm = s;
    if (fork && seen++ > 0) {   // the first track stays on the caller's stream (programmatic launch behind the step kernel)
      if (!env->map_stream[mid]) {
        CUDA_TRY(env, cudaStreamCreateWithFlags(&env->map_stream[mid], cudaStreamNonBlocking));
        CUDA_TRY(env, cudaEventCreateWithFlags(&env->ev_join[mid], cudaEventDisableTiming));
      }
      sm = env->map_stream[mid];
      CUDA_TRY(env, cudaStreamWaitEvent(sm, env->ev_fork, 0));
      forked[mid] = true;
    } else if (fork) {
      // fork point: everything enqueued on `s` so far (the step / reset kernel), NOT the first track's observation kernels
      if (!env->ev_fork) CUDA_TRY(env, cudaEventCreateWithFlags(&env->ev_fork, cudaEventDisableTiming));
      CUDA_TRY(env, cudaEventRecord(env->ev_fork, s));
    }
    env->in_fork = forked[mid];
    if (out->lidar_dev && (env->cfg.obs_flags & RD_OBS_LIDAR)) {
      int rc = launch_lidar(env, mid, env->d_recs, order, n_env, out->lidar_dev, sm, ctr);
      if (rc) { env->in_fork = false; return rc; }
    }
    if (out->occupancy_dev && (env->cfg.obs_flags & RD_OBS_OCCUPANCY)) {
      int rc = launch_occupancy(env, mid, env->d_recs, nullptr, order, n_env, out->occupancy_dev, sm);
      if (rc) { env->in_fork = false; return rc; }
    }
    env->in_fork = false;
    if (forked[mid]) CUDA_TRY(env, cudaEventRecord(env->ev_join[mid], sm));
  }
  for (int mid = 0; mid < RD_MAX_MAPS; ++mid)
    if (forked[mid]) CUDA_TRY(env, cudaStreamWaitEvent(s, env->ev_join[mid], 0));
  return RD_OK;
}

int ensure_stage(rd_env* env, int n) {
  if (n <= env->stage_cap) return RD_OK;
  if (env->d_stage_recs) cudaFree(env->d_stage_recs);
  if (env->d_stage_ids) cudaFree(env->d_stage_ids);
  env->d_stage_recs = nullptr; env->d_stage_ids = nullptr; env->stage_cap = 0;
  CUDA_TRY(env, cudaMalloc(&env->d_stage_recs, sizeof(OriginRec) * (size_t)n));
  CUDA_TRY(env, cudaMalloc(&env->d_stage_ids, sizeof(int32_t) * (size_t)n));
  env->stage_cap = n;
  return RD_OK;
}

// map_ids_host: ascending or NULL.  Fills runs[mid] = (first, count) and uploads the ids.
int stage_runs(rd_env* env, const int32_t* ids, int n, int (*runs)[2], cudaStream_t s) {
  for (int i = 0; i < RD_MAX_MAPS; ++i) runs[i][0] = runs[i][1] = 0;
  if (!ids) {
    if (!env->maps[0].present) return fail(env, RD_ERR_STATE, "map 0 not uploaded");
    runs[0][0] = 0; runs[0][1] = n;
    return RD_OK;
  }
  for (int i = 0; i < n; ++i) {
    const int id = ids[i];
    if (id < 0 || id >= RD_MAX_MAPS || !env->maps[id].present) return fail(env, RD_ERR_INVALID, "map id %d not uploaded", id);
    if (i > 0 && id < ids[i - 1]) return fail(env, RD_ERR_INVALID, "map_ids must be ascending");
    if (runs[id][1] == 0) runs[id][0] = i;
    runs[id][1]++;
  }
  CUDA_TRY(env, cudaMemcpyAsync(env->d_stage_ids, ids, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, s));
  return RD_OK;
}

void store_free(rd_env::Store& st) {
  for (int k = 0; k < SK_N; ++k) cudaFree(st.d.rows[k]);
  cudaFree(st.d.head); cudaFree(st.d.ep_start); cudaFree(st.d.table); cudaFree(st.d.next_id); cudaFree(st.d.fin);
  cudaFree(st.d_all); cudaFree(st.d_invalid); cudaFree(st.d_elig); cudaFree(st.d_n_elig); cudaFree(st.d_cub);
  cudaFree(st.d_req_id); cudaFree(st.d_req_start); cudaFree(st.d_export);
  for (int k = 0; k < SK_N; ++k) cudaFree(st.d.imp[k]);
  cudaFree(st.d.itable); cudaFree(st.d_imp_len); cudaFree(st.d_imp_first);
  st = rd_env::Store{};
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
RD_API void rd_default_config(rd_config* cfg) { if (cfg) default_config(cfg); }
RD_API int rd_abi_version(void) { return RD_ABI_VERSION; }
RD_API const char* rd_last_error(const rd_env* env) { return env ? env->error.c_str() : g_last_error.c_str(); }
RD_API int64_t rd_launch_count(const rd_env* env) { return env ? env->launches : 0; }

RD_API int rd_create(const rd_config* cfg, rd_env** out) {
  if (!cfg || !out) return fail(nullptr, RD_ERR_INVALID, "null argument");
  *out = nullptr;
  if (cfg->abi_version != RD_ABI_VERSION) return fail(nullptr, RD_ERR_INVALID, "abi_version %d != %d", cfg->abi_version, RD_ABI_VERSION);
  if (cfg->n_envs < 1 || cfg->n_beams < 1 || cfg->n_beams > 8192 || cfg->action_repeat < 1 || cfg->n_checkpoints < 1 ||
      !(cfg->dt > 0.0) || !(cfg->lidar_range_max > 0.0))
    return fail(nullptr, RD_ERR_INVALID, "bad config (n_envs %d, n_beams %d, action_repeat %d)", cfg->n_envs, cfg->n_beams, cfg->action_repeat);
  {
    const int A = cfg->agents_per_world;
    if (A > RD_MAX_AGENTS || (A > 1 && cfg->n_envs % A != 0))
      return fail(nullptr, RD_ERR_INVALID, "agents_per_world %d: must be 1..%d and divide n_envs %d", A, RD_MAX_AGENTS, cfg->n_envs);
    bool nstep = A > 1 ? false : cfg->task == RD_TASK_N_STEP_PROGRESS;
    for (int a = 0; a < A && A > 1; ++a) {
      if (cfg->agent_task[a] < RD_TASK_MAX_PROGRESS || cfg->agent_task[a] > RD_TASK_N_STEP_PROGRESS)
        return fail(nullptr, RD_ERR_INVALID, "agent_task[%d] = %d is not an RD_TASK_*", a, cfg->agent_task[a]);
      nstep = nstep || cfg->agent_task[a] == RD_TASK_N_STEP_PROGRESS;
    }
    if (nstep && (cfg->n_step_progress < 1 || cfg->n_step_progress > RD_MAX_NSTEP))
      return fail(nullptr, RD_ERR_INVALID, "n_step_progress %d out of range [1,%d]", cfg->n_step_progress, RD_MAX_NSTEP);
    if (A > 1 && !(cfg->ball_spacing > 0.0)) return fail(nullptr, RD_ERR_INVALID, "ball_spacing must be positive");
    if (cfg->time_limit_ticks < 0) return fail(nullptr, RD_ERR_INVALID, "time_limit_ticks must be >= 0");
    if (cfg->obs_flags & RD_OBS_NORM_BASELINES) {
      if (cfg->obs_flags & RD_OBS_LIDAR_NORM) return fail(nullptr, RD_ERR_INVALID, "RD_OBS_NORM_BASELINES excludes RD_OBS_LIDAR_NORM");
      for (int k = 0; k < 3; ++k)
        if (!(cfg->obs_high[k] > cfg->obs_low[k])) return fail(nullptr, RD_ERR_INVALID, "obs_high[%d] must exceed obs_low[%d]", k, k);
    }
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    cudaGetLastError();
    return fail(nullptr, RD_ERR_NO_DEVICE, "no CUDA device: librd_env has no CPU fallback");
  }
  int dev = 0;
  CUDA_TRY(nullptr, cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CUDA_TRY(nullptr, cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(nullptr, RD_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major, prop.minor);
  rd_env* env = new (std::nothrow) rd_env();
  if (!env) return fail(nullptr, RD_ERR_NOMEM, "out of host memory");
  env->cfg = *cfg;
  env->device = dev;
  env->sm_count = prop.multiProcessorCount;
  env->smem_optin = (int)prop.sharedMemPerBlockOptin;
  env->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  env->n = cfg->n_envs;
  env->order_offset.assign(RD_MAX_MAPS + 1, 0);
  // L2 residency of the tracks (launch_attrs): set aside a slice of L2 for persisting lines, once per device; the
  // slice only ever grows (another handle or the application may have asked for more).
  if (prop.persistingL2CacheMaxSize > 0 && prop.accessPolicyMaxWindowSize > 0) {
    size_t cur = 0;
    const size_t want = std::min<size_t>((size_t)prop.persistingL2CacheMaxSize, (size_t)8 << 20);
    if (cudaDeviceGetLimit(&cur, cudaLimitPersistingL2CacheSize) == cudaSuccess &&
        (cur >= want || cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess))
      env->l2_window_max = std::min<size_t>((size_t)prop.accessPolicyMaxWindowSize, std::max(cur, want));
    cudaGetLastError();
  }
  // k_step is one long float64 instruction stream per warp: spread the warps over as many SM sub-partitions as the
  // batch allows
  env->step_block = (env->n >= 128 * 4 * env->sm_count) ? 128 : ((env->n >= 64 * 4 * env->sm_count) ? 64 : 32);
  if (const char* ev = std::getenv("RD_LIDAR_ORDER")) env->lidar_centre_first = std::atoi(ev) != 0;
  env->step_split = env->n <= 64 * env->sm_count;   // up to two CTAs per SM -- what the kernel's registers allow, a third CTA
                                                     // would wait for a second wave (measured: 22.9 vs 31.9 us at 8192 envs, 39.1 vs
                                                     // 33.0 us at 12 288; rotating the warp roles of co-resident CTAs over the
                                                     // schedulers changes nothing, profiles/r6b_two_tracks_strong_scaling.txt)
  if (const char* ev = std::getenv("RD_STEP_SPLIT")) env->step_split = std::atoi(ev) != 0;
  if (const char* ev = std::getenv("RD_FORK_MAPS")) env->fork_maps = std::atoi(ev) != 0;
  const size_t n = (size_t)env->n;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) { e = cudaMalloc(p, bytes); if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes); } };
  env->vk = rdv_make_const(cfg->vehicle, cfg->dt);
  env->voff = rdv_acc_set(env->vk, 0.0);
  alloc((void**)&env->d_vk, sizeof(VehConst));
  alloc((void**)&env->d_voff, sizeof(VehAcc));
  if (e == cudaSuccess) e = cudaMemcpy(env->d_vk, &env->vk, sizeof(VehConst), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(env->d_voff, &env->voff, sizeof(VehAcc), cudaMemcpyHostToDevice);
  alloc((void**)&env->d_f2, sizeof(double2) * RD_NPAIR * n);
  alloc((void**)&env->d_i4, sizeof(int4) * n);
  alloc((void**)&env->d_i2, sizeof(int2) * n);
  alloc((void**)&env->d_stats, sizeof(double) * 16);
  alloc((void**)&env->d_recs, sizeof(OriginRec) * n);
  {
    const int A = cfg->agents_per_world > 1 ? cfg->agents_per_world : 1;
    bool nstep = A > 1 ? false : cfg->task == RD_TASK_N_STEP_PROGRESS;
    for (int a = 0; a < A && A > 1; ++a) nstep = nstep || cfg->agent_task[a] == RD_TASK_N_STEP_PROGRESS;
    env->multi = A > 1 || nstep;
    if (nstep) alloc((void**)&env->d_hist, sizeof(double) * (size_t)cfg->n_step_progress * n);
  }
  alloc((void**)&env->d_beam_tab, sizeof(double) * 2 * (size_t)cfg->n_beams);
  alloc((void**)&env->d_maps, sizeof(DevMap) * RD_MAX_MAPS);
  alloc((void**)&env->d_env_order, sizeof(int32_t) * n);
  alloc((void**)&env->d_lidar_ctr, sizeof(unsigned int) * 2 * RD_CTR_RING);
  if (e != cudaSuccess) {
    int rc = fail(nullptr, e == cudaErrorMemoryAllocation ? RD_ERR_NOMEM : RD_ERR_CUDA, "allocation: %s", cudaGetErrorString(e));
    rd_destroy(env);
    return rc;
  }
  // beam table: angle_i = fov/2 - i*fov/(n-1) [REF dreamer/tools.py:84-86], float64 cos | sin
  std::vector<double> tab(2 * (size_t)cfg->n_beams);
  for (int i = 0; i < cfg->n_beams; ++i) {
    double a = (cfg->n_beams > 1) ? (0.5 * cfg->lidar_fov - (double)i * (cfg->lidar_fov / (double)(cfg->n_beams - 1))) : 0.0;
    tab[i] = std::cos(a);
    tab[cfg->n_beams + i] = std::sin(a);
  }
  e = cudaMemcpy(env->d_beam_tab, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { int rc = fail(nullptr, RD_ERR_CUDA, "beam table upload: %s", cudaGetErrorString(e)); rd_destroy(env); return rc; }
  *out = env;
  return RD_OK;
}

RD_API void rd_destroy(rd_env* env) {
  if (!env) return;
  cudaFree(env->d_vk); cudaFree(env->d_voff);
  cudaFree(env->d_f2); cudaFree(env->d_i4); cudaFree(env->d_i2); cudaFree(env->d_stats); cudaFree(env->d_hist); cudaFree(env->d_recs);
  cudaFree(env->d_beam_tab); cudaFree(env->d_maps); cudaFree(env->d_env_order); cudaFree(env->d_lidar_ctr);
  cudaFree(env->d_stage_recs); cudaFree(env->d_stage_ids);
  cudaFree(env->pol.st.f64); cudaFree(env->pol.st.i32); cudaFree(env->pol.d_actions);
  dreamer_free(env->dr);
  store_free(env->st);
  occ_free(env->occ);
  {
    auto& h = env->hp;
    for (auto st : h.streams) cudaStreamDestroy(st);
    for (auto ev : h.ev_done) cudaEventDestroy(ev);
    if (h.ev_act) cudaEventDestroy(h.ev_act);
    cudaFreeHost(h.act_host); cudaFree(h.act_dev); cudaFree(h.mask_dev); cudaFree(h.small_dev); cudaFreeHost(h.small_host);
    cudaFree(h.lidar_dev); cudaFreeHost(h.lidar_host); cudaFree(h.occ_dev); cudaFreeHost(h.occ_host);
  }
  for (auto& t : env->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
  for (auto& e : env->event_pool) cudaEventDestroy(e);
  for (int mid = 0; mid < RD_MAX_MAPS; ++mid) {
    if (env->map_stream[mid]) cudaStreamDestroy(env->map_stream[mid]);
    if (env->ev_join[mid]) cudaEventDestroy(env->ev_join[mid]);
  }
  if (env->ev_fork) cudaEventDestroy(env->ev_fork);
  for (auto& m : env->maps) { cudaFree(m.d_bits); cudaFree(m.d_dist); cudaFree(m.d_start); cudaFree(m.d_reset); cudaFree(m.d_next); }
  delete env;
}

RD_API int rd_upload_map(rd_env* env, int map_id, const uint32_t* bits_host, int h, int w, int row_words,
                         const uint16_t* dist_host, int dmax, double resolution, double origin_x, double origin_y,
                         int col0, int row0_yup, int full_h, const double* start_poses_host, int n_start,
                         const double* reset_poses_host, int n_reset) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (map_id < 0 || map_id >= RD_MAX_MAPS) return fail(env, RD_ERR_INVALID, "map_id %d out of range [0,%d)", map_id, RD_MAX_MAPS);
  if (!bits_host || !dist_host || !start_poses_host || h < 3 || w < 3 || row_words * 32 < w || n_start < 1 || dmax < 1 || !(resolution > 0.0))
    return fail(env, RD_ERR_INVALID, "bad map arguments");
  // the ray march relies on a non-drivable border: verify it instead of trusting the caller
  for (int x = 0; x < w; ++x) {
    if (((bits_host[(size_t)0 * row_words + (x >> 5)] >> (x & 31)) & 1u) || ((bits_host[(size_t)(h - 1) * row_words + (x >> 5)] >> (x & 31)) & 1u))
      return fail(env, RD_ERR_INVALID, "map %d: border row has drivable cells", map_id);
  }
  for (int y = 0; y < h; ++y) {
    const uint32_t* row = bits_host + (size_t)y * row_words;
    if ((row[0] & 1u) || ((row[(w - 1) >> 5] >> ((w - 1) & 31)) & 1u)) return fail(env, RD_ERR_INVALID, "map %d: border column has drivable cells", map_id);
    for (int x = w; x < row_words * 32; ++x)
      if ((row[x >> 5] >> (x & 31)) & 1u) return fail(env, RD_ERR_INVALID, "map %d: padding bits set", map_id);
  }
  HostMap& m = env->maps[map_id];
  cudaFree(m.d_bits); cudaFree(m.d_dist); cudaFree(m.d_start); cudaFree(m.d_reset); cudaFree(m.d_next);
  m = HostMap{};
  const size_t bits_bytes = (size_t)h * row_words * 4;
  const size_t bits_padded = (bits_bytes + 15) & ~(size_t)15;
  // block clearance field for the ray march's empty-space skipping (rd_march.cuh), stored right behind the bits so
  // that one bulk copy brings both into shared memory
  std::vector<uint8_t> coarse;
  int ch = 0, cw = 0;
  // Block size of the clearance field: the finest that still fits in shared memory next to the bits and the beam
  // table.  Measured on B200: 2x2 blocks beat 4x4 by 10-13 % even where they halve the resident warps (fewer exact-DDA
  // steps at the end of each ray matter more than occupancy).
  int cshift = 1;
  const size_t fixed = 16 + (((size_t)2 * env->cfg.n_beams * 8 + 15) & ~(size_t)15) + bits_padded;
  while (cshift < 5 && fixed + (size_t)(((h >> cshift) + 1) * ((w >> cshift) + 1)) + 16 > (size_t)env->smem_optin) ++cshift;
  rd_build_clearance(bits_host, h, w, row_words, cshift, coarse, ch, cw);
  const size_t coarse_padded = (coarse.size() + 15) & ~(size_t)15;
  std::vector<unsigned char> packed(bits_padded + coarse_padded, 0);
  std::memcpy(packed.data(), bits_host, bits_bytes);
  std::memcpy(packed.data() + bits_padded, coarse.data(), coarse.size());
  // the two arrays every step reads (bit grid + clearance field, wavefront distance) share ONE allocation, so that a
  // single L2 access-policy window can keep the whole track resident (launch_attrs)
  const size_t dist_off = (packed.size() + 255) & ~(size_t)255, dist_bytes = sizeof(uint16_t) * (size_t)h * w;
  CUDA_TRY(env, cudaMalloc(&m.d_bits, dist_off + dist_bytes));
  CUDA_TRY(env, cudaMemcpy(m.d_bits, packed.data(), packed.size(), cudaMemcpyHostToDevice));
  void* dist_dev = static_cast<unsigned char*>(m.d_bits) + dist_off;
  CUDA_TRY(env, cudaMemcpy(dist_dev, dist_host, dist_bytes, cudaMemcpyHostToDevice));
  m.hot_bytes = dist_off + dist_bytes;
  CUDA_TRY(env, cudaMalloc(&m.d_start, sizeof(double) * 3 * (size_t)n_start));
  CUDA_TRY(env, cudaMemcpy(m.d_start, start_poses_host, sizeof(double) * 3 * (size_t)n_start, cudaMemcpyHostToDevice));
  if (n_reset > 0 && reset_poses_host) {
    CUDA_TRY(env, cudaMalloc(&m.d_reset, sizeof(double) * 3 * (size_t)n_reset));
    CUDA_TRY(env, cudaMemcpy(m.d_reset, reset_poses_host, sizeof(double) * 3 * (size_t)n_reset, cudaMemcpyHostToDevice));
  } else {
    n_reset = 0;
  }
  DevMap& d = m.dev;
  d.bits = (const uint32_t*)m.d_bits; d.dist = (const uint16_t*)dist_dev;
  d.start = (const double*)m.d_start; d.reset = (const double*)m.d_reset;
  d.h = h; d.w = w; d.rw = row_words; d.col0 = col0; d.row0 = row0_yup; d.full_h = full_h; d.dmax = dmax;
  d.n_start = n_start; d.n_reset = n_reset; d.bits_bytes = (int)packed.size();
  d.coarse_off = (int)bits_padded; d.cw = cw; d.ch = ch; d.cshift = cshift;
  d.res = resolution; d.inv_res = 1.0 / resolution; d.ox = origin_x; d.oy = origin_y;
  d.inv_dmax = 1.0 / (double)dmax;
  if (n_reset > 0) {
    // random_ball chain: next[i] = the reset pose with the smallest wavefront distance that is at least
    // ceil(ball_spacing / resolution) cells of progress beyond pose i, wrapping over the finish line.  The wavefront
    // distance is a Chebyshev path length, so consecutive cars of a world stand at least ball_spacing metres apart.
    std::vector<int32_t> dpose(n_reset), next(n_reset);
    std::vector<std::pair<int32_t, int32_t>> key(n_reset);
    for (int i = 0; i < n_reset; ++i) {
      const double u = (reset_poses_host[3 * i] - origin_x) * d.inv_res, v = (reset_poses_host[3 * i + 1] - origin_y) * d.inv_res;
      const double fu = std::floor(u), fv = std::floor(v);
      int32_t dv = 0;
      if (fu > -1.0e9 && fu < 1.0e9 && fv > -1.0e9 && fv < 1.0e9) {
        const int cx = (int)fu - col0, cy = (int)fv - row0_yup;
        if (cx >= 0 && cx < w && cy >= 0 && cy < h) dv = (int32_t)dist_host[(size_t)cy * w + cx];
      }
      dpose[i] = dv;
      key[i] = {dv, i};
    }
    std::sort(key.begin(), key.end());
    const int32_t sc = (int32_t)std::ceil(env->cfg.ball_spacing / resolution);
    auto first_at_least = [&](int32_t dv) { return (int)(std::lower_bound(key.begin(), key.end(), std::make_pair(dv, (int32_t)INT32_MIN)) - key.begin()); };
    for (int i = 0; i < n_reset; ++i) {
      int j = first_at_least(dpose[i] + sc);
      if (j == n_reset) j = first_at_least(dpose[i] + sc - dmax);
      next[i] = j < n_reset ? key[j].second : i;
    }
    CUDA_TRY(env, cudaMalloc(&m.d_next, sizeof(int32_t) * (size_t)n_reset));
    CUDA_TRY(env, cudaMemcpy(m.d_next, next.data(), sizeof(int32_t) * (size_t)n_reset, cudaMemcpyHostToDevice));
    d.ball_next = (const int32_t*)m.d_next;
  }
  m.present = true;
  env->maps_dirty = true;
  return RD_OK;
}

RD_API int rd_assign_maps(rd_env* env, const int32_t* ids) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  const int n = env->n;
  std::vector<int32_t> id(n, 0);
  if (ids) std::copy(ids, ids + n, id.begin());
  std::vector<int> count(RD_MAX_MAPS, 0);
  for (int e = 0; e < n; ++e) {
    if (id[e] < 0 || id[e] >= RD_MAX_MAPS || !env->maps[id[e]].present) return fail(env, RD_ERR_INVALID, "env %d: map id %d not uploaded", e, id[e]);
    count[id[e]]++;
    const int A = env->cfg.agents_per_world;
    if (A > 1 && id[e] != id[e - e % A]) return fail(env, RD_ERR_INVALID, "env %d: the cars of one world must share a map", e);
  }
  env->order_offset[0] = 0;
  for (int m = 0; m < RD_MAX_MAPS; ++m) env->order_offset[m + 1] = env->order_offset[m] + count[m];
  std::vector<int> cursor(env->order_offset.begin(), env->order_offset.end() - 1);
  std::vector<int32_t> order(n);
  for (int e = 0; e < n; ++e) order[cursor[id[e]]++] = e;
  CUDA_TRY(env, cudaMemcpy(env->d_env_order, order.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice));
  env->h_order = order;
  CUDA_TRY(env, cudaMemcpy2D(reinterpret_cast<int32_t*>(env->d_i2) + 1, sizeof(int2), id.data(), sizeof(int32_t), sizeof(int32_t),
                             (size_t)n, cudaMemcpyHostToDevice));   // the .y (map) column of the (episode, map) group
  int rc = sync_maps(env);
  if (rc) return rc;
  env->assigned = true;
  return RD_OK;
}

RD_API int rd_reset(rd_env* env, const uint8_t* mask_dev, int mode, const rd_outputs* out, void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (!env->assigned) return fail(env, RD_ERR_STATE, "rd_assign_maps has not been called");
  if (mode < RD_RESET_GRID || mode > RD_RESET_RANDOM_BALL) return fail(env, RD_ERR_INVALID, "bad reset mode %d", mode);
  int rc = sync_maps(env);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  {
    ScopedTiming tm(env, s, T_RESET);
    k_reset<<<(env->n + 127) / 128, 128, 0, s>>>(step_params(env), out_ptrs(out), mask_dev, mode, 0);
  }
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  env->was_reset = true;
  return observe(env, out, s, 0, -1, nullptr, true);
}

RD_API int rd_step(rd_env* env, const float* actions_dev, const rd_outputs* out, void* stream) {
  if (!env || !actions_dev) return fail(env, RD_ERR_INVALID, "null argument");
  if (!env->assigned) return fail(env, RD_ERR_STATE, "rd_assign_maps has not been called");
  if (!env->was_reset) return fail(env, RD_ERR_STATE, "Must reset environment.");  // [REF dreamer/wrappers.py:148]
  cudaStream_t s = (cudaStream_t)stream;
  int rc = launch_step(env, out, actions_dev, s);
  if (rc) return rc;
  return observe(env, out, s, 0, -1, nullptr, true);
}

// ---------------------------------------------------------------------------------------------------------
// host-facing path
RD_API int rd_host_init(rd_env* env, int n_chunks, rd_outputs* host_out) {
  if (!env || !host_out) return fail(env, RD_ERR_INVALID, "null argument");
  if (!env->assigned) return fail(env, RD_ERR_STATE, "rd_assign_maps has not been called");
  auto& h = env->hp;
  if (h.ready) { *host_out = h.host_out; return RD_OK; }
  const int n = env->n;
  n_chunks = std::max(1, std::min(n_chunks, n));
  h.n_chunks = n_chunks;
  // progressive chunk sizes (1 : 2 : 4 : ... capped at 16x, measured with the round-2 kernels): the first chunk is small so that the copy engine starts
  // early; from then on it is the bottleneck and each chunk's ray casting hides behind the previous chunk's copy.
  {
    auto weight = [](int c) { return (double)(1 << std::min(c, 4)); };
    h.bounds.assign(n_chunks + 1, 0);
    double tot = 0.0, acc = 0.0;
    for (int c = 0; c < n_chunks; ++c) tot += weight(c);
    for (int c = 0; c < n_chunks; ++c) { acc += weight(c); h.bounds[c + 1] = (int)std::llround((double)n * acc / tot); }
    h.bounds[n_chunks] = n;
  }
  // small arrays share one slab (one device->host copy per step); offsets 256-byte aligned
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
  const size_t o_pose = take(sizeof(float) * 6 * n), o_vel = take(sizeof(float) * 6 * n), o_speed = take(sizeof(float) * n);
  const size_t o_rew = take(sizeof(float) * n), o_prog = take(sizeof(float) * n), o_time = take(sizeof(float) * n);
  const size_t o_lap = take(sizeof(int32_t) * n), o_done = take((size_t)n), o_flags = take((size_t)n);
  const size_t o_rank = take(sizeof(int32_t) * n), o_opp = take((size_t)n);
  const size_t o_ww = take((size_t)n), o_wc = take((size_t)n);
  h.small_bytes = off;
  const size_t lidar_elem = (env->cfg.obs_flags & RD_OBS_LIDAR_F16) ? 2 : 4;
  h.lidar_elem = lidar_elem;
  const size_t lidar_bytes = lidar_elem * (size_t)n * env->cfg.n_beams;
  const bool occ = (env->cfg.obs_flags & RD_OBS_OCCUPANCY) != 0;
  CUDA_TRY(env, cudaMalloc(&h.small_dev, h.small_bytes));
  CUDA_TRY(env, cudaMemset(h.small_dev, 0, h.small_bytes));
  CUDA_TRY(env, cudaHostAlloc(&h.small_host, h.small_bytes, cudaHostAllocDefault));
  std::memset(h.small_host, 0, h.small_bytes);
  CUDA_TRY(env, cudaHostAlloc(&h.lidar_host, lidar_bytes, cudaHostAllocDefault));
  std::memset(h.lidar_host, 0, lidar_bytes);
  CUDA_TRY(env, cudaMalloc(&h.lidar_dev, lidar_bytes));
  CUDA_TRY(env, cudaMemset(h.lidar_dev, 0, lidar_bytes));
  if (occ) {
    CUDA_TRY(env, cudaMalloc(&h.occ_dev, (size_t)n * 4096));
    CUDA_TRY(env, cudaMemset(h.occ_dev, 0, (size_t)n * 4096));
    CUDA_TRY(env, cudaHostAlloc(&h.occ_host, (size_t)n * 4096, cudaHostAllocDefault));
    std::memset(h.occ_host, 0, (size_t)n * 4096);
  }
  CUDA_TRY(env, cudaHostAlloc(&h.act_host, sizeof(float) * 2 * n, cudaHostAllocDefault));
  CUDA_TRY(env, cudaMalloc(&h.act_dev, sizeof(float) * 2 * n));
  CUDA_TRY(env, cudaMalloc(&h.mask_dev, (size_t)n));
  h.streams.resize(n_chunks);
  h.ev_done.resize(n_chunks);
  for (int c = 0; c < n_chunks; ++c) {
    CUDA_TRY(env, cudaStreamCreateWithFlags(&h.streams[c], cudaStreamNonBlocking));
    CUDA_TRY(env, cudaEventCreateWithFlags(&h.ev_done[c], cudaEventDisableTiming));
  }
  CUDA_TRY(env, cudaEventCreateWithFlags(&h.ev_act, cudaEventDisableTiming));
  auto fill = [&](rd_outputs& o, unsigned char* base, float* lidar, uint8_t* occp) {
    o.lidar_dev = lidar; o.occupancy_dev = occp;
    o.pose_dev = (float*)(base + o_pose); o.velocity_dev = (float*)(base + o_vel); o.speed_dev = (float*)(base + o_speed);
    o.reward_dev = (float*)(base + o_rew); o.progress_dev = (float*)(base + o_prog); o.time_dev = (float*)(base + o_time);
    o.lap_dev = (int32_t*)(base + o_lap); o.done_dev = (uint8_t*)(base + o_done); o.flags_dev = (uint8_t*)(base + o_flags);
    o.rank_dev = (int32_t*)(base + o_rank); o.opponents_dev = (uint8_t*)(base + o_opp);
    o.wrong_way_dev = (uint8_t*)(base + o_ww); o.wall_collision_dev = (uint8_t*)(base + o_wc);
  };
  fill(h.dev_out, h.small_dev, h.lidar_dev, h.occ_dev);
  fill(h.host_out, h.small_host, h.lidar_host, h.occ_host);
  h.ready = true;
  *host_out = h.host_out;
  return RD_OK;
}

namespace {
// makes the handle's device current for the duration of a host-facing call
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
// device->host copies of the chunk's big rows on its stream; the last step of the call gathers the small slab
int host_copy_back(rd_env* env, int c) {
  auto& h = env->hp;
  const size_t e0 = (size_t)h.bounds[c], cnt = (size_t)(h.bounds[c + 1] - h.bounds[c]);
  const size_t nb = (size_t)env->cfg.n_beams;
  const size_t off = e0 * nb * h.lidar_elem;
  CUDA_TRY(env, cudaMemcpyAsync(reinterpret_cast<unsigned char*>(h.lidar_host) + off, reinterpret_cast<unsigned char*>(h.lidar_dev) + off,
                                h.lidar_elem * cnt * nb, cudaMemcpyDeviceToHost, h.streams[c]));
  if (h.occ_dev) CUDA_TRY(env, cudaMemcpyAsync(h.occ_host + e0 * 4096, h.occ_dev + e0 * 4096, cnt * 4096, cudaMemcpyDeviceToHost, h.streams[c]));
  return RD_OK;
}
// joins every chunk stream into stream 0 (and, `wait`, blocks until the results are in the host buffers)
int host_finish(rd_env* env, bool small_copied, bool wait = true) {
  auto& h = env->hp;
  for (int c = 1; c < h.n_chunks; ++c) {
    CUDA_TRY(env, cudaEventRecord(h.ev_done[c], h.streams[c]));
    CUDA_TRY(env, cudaStreamWaitEvent(h.streams[0], h.ev_done[c], 0));
  }
  if (!small_copied) CUDA_TRY(env, cudaMemcpyAsync(h.small_host, h.small_dev, h.small_bytes, cudaMemcpyDeviceToHost, h.streams[0]));
  if (wait) CUDA_TRY(env, cudaStreamSynchronize(h.streams[0]));
  return RD_OK;
}
}  // namespace

RD_API int rd_reset_host(rd_env* env, const uint8_t* mask_host, int mode) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  auto& h = env->hp;
  if (!h.ready) return fail(env, RD_ERR_STATE, "rd_host_init has not been called");
  if (h.pending) return fail(env, RD_ERR_STATE, "rd_step_host_begin is pending: call rd_step_host_end first");
  DeviceGuard guard(env->device);
  cudaStream_t s0 = h.streams[0];
  if (mask_host) CUDA_TRY(env, cudaMemcpyAsync(h.mask_dev, mask_host, (size_t)env->n, cudaMemcpyHostToDevice, s0));
  int rc = rd_reset(env, mask_host ? h.mask_dev : nullptr, mode, &h.dev_out, s0);
  if (rc) return rc;
  const int saved = h.n_chunks;   // everything ran on stream 0: copy it back as one chunk
  const size_t nb = (size_t)env->cfg.n_beams, n = (size_t)env->n;
  CUDA_TRY(env, cudaMemcpyAsync(h.lidar_host, h.lidar_dev, h.lidar_elem * n * nb, cudaMemcpyDeviceToHost, s0));
  if (h.occ_dev) CUDA_TRY(env, cudaMemcpyAsync(h.occ_host, h.occ_dev, n * 4096, cudaMemcpyDeviceToHost, s0));
  CUDA_TRY(env, cudaMemcpyAsync(h.small_host, h.small_dev, h.small_bytes, cudaMemcpyDeviceToHost, s0));
  CUDA_TRY(env, cudaStreamSynchronize(s0));
  (void)saved;
  return RD_OK;
}

namespace { int step_host_enqueue(rd_env* env, const float* actions_host, bool wait); }

RD_API int rd_step_host(rd_env* env, const float* actions_host) {
  if (env && env->hp.pending) return fail(env, RD_ERR_STATE, "rd_step_host_begin is pending: call rd_step_host_end first");
  return step_host_enqueue(env, actions_host, true);
}

RD_API int rd_step_host_begin(rd_env* env, const float* actions_host) {
  if (env && env->hp.pending) return fail(env, RD_ERR_STATE, "rd_step_host_begin is pending: call rd_step_host_end first");
  int rc = step_host_enqueue(env, actions_host, false);
  if (rc == RD_OK) env->hp.pending = true;
  return rc;
}

RD_API int rd_step_host_end(rd_env* env) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  auto& h = env->hp;
  if (!h.ready || !h.pending) return fail(env, RD_ERR_STATE, "no rd_step_host_begin is pending");
  DeviceGuard guard(env->device);
  h.pending = false;
  CUDA_TRY(env, cudaStreamSynchronize(h.streams[0]));
  return RD_OK;
}

namespace {
int step_host_enqueue(rd_env* env, const float* actions_host, bool wait) {
  if (!env || !actions_host) return fail(env, RD_ERR_INVALID, "null argument");
  auto& h = env->hp;
  if (!h.ready) return fail(env, RD_ERR_STATE, "rd_host_init has not been called");
  if (!env->was_reset) return fail(env, RD_ERR_STATE, "Must reset environment.");  // [REF dreamer/wrappers.py:148]
  DeviceGuard guard(env->device);
  const int n = env->n;
  std::memcpy(h.act_host, actions_host, sizeof(float) * 2 * (size_t)n);   // caller memory may be pageable
  CUDA_TRY(env, cudaMemcpyAsync(h.act_dev, h.act_host, sizeof(float) * 2 * (size_t)n, cudaMemcpyHostToDevice, h.streams[0]));
  // k_step is bound by the latency of one env's float64 dependency chain, not by the batch size, so it runs ONCE
  // over the whole batch; the observation kernels then go chunk by chunk so that chunk k's device->host copy
  // overlaps chunk k+1's ray casting.  The small result slab is copied right behind k_step.
  cudaStream_t s0 = h.streams[0];
  if (int rc = launch_step(env, &h.dev_out, h.act_dev, s0)) return rc;
  CUDA_TRY(env, cudaEventRecord(h.ev_act, s0));   // marks "state advanced"
  bool small_copied = false;
  for (int c = 0; c < h.n_chunks; ++c) {
    cudaStream_t s = h.streams[c];
    const int e0 = h.bounds[c], e1 = h.bounds[c + 1];
    if (e1 <= e0) continue;
    if (c > 0) CUDA_TRY(env, cudaStreamWaitEvent(s, h.ev_act, 0));
    if (c == 1) {  // the small slab is final once k_step is done: copy it while chunk 0 is ray casting
      CUDA_TRY(env, cudaMemcpyAsync(h.small_host, h.small_dev, h.small_bytes, cudaMemcpyDeviceToHost, s));
      small_copied = true;
    }
    int rc = observe(env, &h.dev_out, s, e0, e1);
    if (rc) return rc;
    if ((rc = host_copy_back(env, c))) return rc;
  }
  return host_finish(env, small_copied, wait);
}
}  // namespace

// ---------------------------------------------------------------------------------------------------------
// on-device policies
RD_API void rd_gap_follower_defaults(const rd_config* cfg, rd_gap_follower* g) {
  if (!cfg || !g) return;
  std::memset(g, 0, sizeof(*g));
  const double deg = 3.14159265358979323846 / 180.0;
  // constants of the node [REF ros_agent/agents/follow_the_gap/src/agent.py:73-104]
  const double max_speed = 7.0, max_decel = 8.26;
  g->lookahead = 2.0 * ((max_speed * max_speed) / (2.0 * max_decel));
  g->vehicle_width = 0.3302 * 1.2;
  g->minimum_gap_length = 0.2;
  g->median_dev_threshold = 9.0;
  g->kp = 1.4; g->ki = 0.0; g->kd = 0.1;
  g->max_vehicle_speed = 6.0;
  g->max_steering_angle = 24.0 * deg;
  g->speed_limit_angle = 5.0 * deg;
  g->scan_dt = (double)cfg->action_repeat * cfg->dt;
  // the scan as a LaserScan message: angle_min = -fov/2, increment = fov/(n-1) [REF dreamer/tools.py:84-86]
  g->angle_min = -0.5 * cfg->lidar_fov;
  g->angle_increment = cfg->n_beams > 1 ? cfg->lidar_fov / (double)(cfg->n_beams - 1) : 1.0;
  g->range_max = cfg->lidar_range_max;
  // get_lidar_scan_arc(-90 deg, +90 deg): int((angle - angle_min) / increment) [REF agent.py:117-126]
  const double a0 = -90.0 * deg, a1 = 90.0 * deg;
  g->arc_first = (int32_t)((a0 - g->angle_min) / g->angle_increment);
  g->arc_last = (int32_t)((a1 - g->angle_min) / g->angle_increment);
  g->filter_width = (int32_t)((10.0 * deg) / g->angle_increment);
  // np.percentile(adjusted, q = 100 * (1 - deg2rad(30) / (a1 - a0))), method 'linear'
  const double q = 100.0 * (1.0 - ((30.0 * deg) / (a1 - a0)));
  const double quant = q / 100.0;
  const int m = g->arc_last - g->arc_first + 1;
  const double vi = (double)m * quant + (1.0 + quant * (1.0 - 1.0 - 1.0)) - 1.0;
  int lo = (int)std::floor(vi);
  g->pct_gamma = vi - (double)lo;
  g->pct_lo = std::min(std::max(lo, 0), m - 1);
  g->pct_hi = std::min(std::max(lo + 1, 0), m - 1);
  g->speed_scale = 0.5;
  g->speed_gain = 1.0;
}

namespace {
// the [n][2] actions the rollouts of every on-device policy write when the caller passes none (one per handle)
int ensure_rollout_actions(rd_env* env) {
  if (env->pol.d_actions) return RD_OK;
  CUDA_TRY(env, cudaMalloc(&env->pol.d_actions, sizeof(float) * 2 * (size_t)env->n));
  CUDA_TRY(env, cudaMemset(env->pol.d_actions, 0, sizeof(float) * 2 * (size_t)env->n));
  return RD_OK;
}
}  // namespace

RD_API int rd_policy_gap_follower_init(rd_env* env, const rd_gap_follower* g_or_null) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (env->cfg.obs_flags & RD_OBS_LIDAR_F16) return fail(env, RD_ERR_INVALID, "the on-device policies read float32 scans: RD_OBS_LIDAR_F16 is set");
  rd_gap_follower g;
  if (g_or_null) g = *g_or_null; else rd_gap_follower_defaults(&env->cfg, &g);
  const int m = g.arc_last - g.arc_first + 1;
  if (g.arc_first < 0 || g.arc_last >= env->cfg.n_beams || m < 8 || g.filter_width < 1 || 2 * g.filter_width >= m ||
      g.pct_lo < 0 || g.pct_hi < g.pct_lo || g.pct_hi >= m || !(g.scan_dt > 0.0) || !(g.angle_increment > 0.0))
    return fail(env, RD_ERR_INVALID, "bad gap-follower parameters (arc %d..%d of %d beams, filter width %d)", g.arc_first,
                g.arc_last, env->cfg.n_beams, g.filter_width);
  if (env->cfg.obs_flags & RD_OBS_LIDAR_NORM) return fail(env, RD_ERR_INVALID, "the gap follower reads ranges in metres (RD_OBS_LIDAR_NORM is set)");
  auto& p = env->pol;
  const size_t n = (size_t)env->n;
  if (!p.st.f64) {
    CUDA_TRY(env, cudaMalloc(&p.st.f64, sizeof(double) * RD_NP_F64 * n));
    CUDA_TRY(env, cudaMalloc(&p.st.i32, sizeof(int32_t) * RD_NP_I32 * n));
  }
  if (int rc = ensure_rollout_actions(env)) return rc;
  std::vector<double> f(RD_NP_F64 * n, 0.0);
  for (size_t e = 0; e < n; ++e) f[(size_t)RD_P_PREV * n + e] = std::nan("");
  CUDA_TRY(env, cudaMemcpy(p.st.f64, f.data(), sizeof(double) * f.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(env, cudaMemset(p.st.i32, 0, sizeof(int32_t) * RD_NP_I32 * n));
  p.g = g;
  p.ready = true;
  return RD_OK;
}

namespace {
int launch_gap_follower(rd_env* env, const float* lidar_dev, const float* speed_dev, float* actions_dev, double* debug_dev,
                        cudaStream_t s) {
  constexpr int WARPS = 8;
  auto& p = env->pol;
  GapArgs A{};
  A.g = p.g; A.ps = p.st; A.lidar = lidar_dev; A.speed = speed_dev; A.state_sv = env->d_f2 + (size_t)RD_P_SV * env->n;
  A.actions = actions_dev; A.debug = debug_dev; A.n = env->n; A.n_beams = env->cfg.n_beams;
  const int m = p.g.arc_last - p.g.arc_first + 1;
  A.m_pad = (m + 1) | 1;   // odd number of floats per row: the warps' rows start in different banks
  A.rescale = env->cfg.rescale_actions;
  for (int k = 0; k < 2; ++k) { A.low[k] = env->cfg.action_low[k]; A.high[k] = env->cfg.action_high[k]; }
  A.a_drive = env->cfg.vehicle.a_drive; A.c_drag = env->cfg.vehicle.c_drag;
  A.steer_scale = env->cfg.vehicle.steer_gain * env->cfg.vehicle.steer_max;
  const size_t smem = sizeof(float) * 2 * (size_t)A.m_pad * WARPS;
  if (smem > (size_t)env->smem_optin || m > 32 * 64) return fail(env, RD_ERR_INVALID, "scan arc of %d beams is too long for the gap follower (max 2048)", m);
  const unsigned grid = (unsigned)((env->n + WARPS - 1) / WARPS);
  auto kern = (m <= 32 * 23) ? k_gap_follower<WARPS, 23>          // 1080 beams: 721 in the arc
              : (m <= 32 * 32) ? k_gap_follower<WARPS, 32> : k_gap_follower<WARPS, 64>;
  if (smem > 48 * 1024 && !env->pol.attr_set) {
    CUDA_TRY(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, env->smem_optin));
    env->pol.attr_set = true;
  }
  {
    ScopedTiming tm(env, s, T_POLICY);
    kern<<<grid, WARPS * 32, smem, s>>>(A);
  }
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}
}  // namespace

RD_API int rd_policy_gap_follower(rd_env* env, const float* lidar_dev, const float* speed_dev, float* actions_dev,
                                  double* debug_dev, void* stream) {
  if (!env || !lidar_dev || !actions_dev) return fail(env, RD_ERR_INVALID, "null argument");
  if (!env->pol.ready) return fail(env, RD_ERR_STATE, "rd_policy_gap_follower_init has not been called");
  return launch_gap_follower(env, lidar_dev, speed_dev, actions_dev, debug_dev, (cudaStream_t)stream);
}

RD_API int rd_rollout_gap_follower(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, void* stream) {
  if (!env || !out || !out->lidar_dev || n_steps < 0) return fail(env, RD_ERR_INVALID, "bad argument (the rollout needs out->lidar_dev)");
  if (!env->pol.ready) return fail(env, RD_ERR_STATE, "rd_policy_gap_follower_init has not been called");
  if (!env->was_reset) return fail(env, RD_ERR_STATE, "Must reset environment.");
  float* act = actions_dev ? actions_dev : env->pol.d_actions;
  for (int k = 0; k < n_steps; ++k) {
    int rc = launch_gap_follower(env, out->lidar_dev, nullptr, act, nullptr, (cudaStream_t)stream);
    if (rc) return rc;
    if ((rc = rd_step(env, act, out, stream))) return rc;
  }
  return RD_OK;
}

namespace {
// training: Dreamer.policy(training=True) -- one sample + exploration (k_actor_train), and each agent's env-step counter
// of the exploration schedule advances by (its envs) x action_repeat [REF dreamer/dreamer.py, Dreamer.__call__ self._step]
int launch_dreamer(rd_env* env, const void* obs_dev, float* actions_dev, int noise, const float* eps_stoch_dev,
                   const float* eps_actor_dev, float* debug_dev, cudaStream_t s, bool training = false,
                   const float* eps_expl_dev = nullptr) {
  int launched = 0, rc;
  DrTrain tr{eps_expl_dev, {}};
  for (int a = 0; a < env->dr.n_agents; ++a) tr.amount.a[a] = dreamer_expl_amount(env->dr, a);
  {
    ScopedTiming tm(env, s, T_POLICY);
    rc = dreamer_step(env->dr, obs_dev, actions_dev, noise, eps_stoch_dev, eps_actor_dev, debug_dev, env->cfg.seed,
                      (uint32_t)env->cfg.env_id_offset, s, &launched, training ? &tr : nullptr);
  }
  env->launches += launched;
  if (rc) return fail(env, rc, "rd_policy_dreamer: %s", env->dr.err.c_str());
  for (int a = 0; training && a < env->dr.n_agents; ++a) env->dr.expl[a].env_steps += (int64_t)env->dr.n_of[a] * env->cfg.action_repeat;
  return RD_OK;
}
// the entry point's agent kind (encoder: the occupancy entry points) must be the initialised agent's
int dreamer_kind(rd_env* env, bool encoder, const char* fn) {
  if (!env->dr.ready) return fail(env, RD_ERR_STATE, "%s: rd_policy_dreamer_init has not been called", fn);
  if (encoder && !env->dr.depth)
    return fail(env, RD_ERR_INVALID, "%s: the agent reads lidar (rd_policy_dreamer_init); use the lidar entry points", fn);
  if (!encoder && env->dr.depth)
    return fail(env, RD_ERR_INVALID, "%s: the agent reads lidar_occupancy (rd_policy_dreamer_init_occupancy); use the "
                "occupancy entry points", fn);
  return RD_OK;
}
// rd_policy_dreamer_init, _init_occupancy (encoder: the latter, enc its image encoder) and _init_agents (G agents:
// w[G], enc[G] or null, agent_of_env [n])
int init_dreamer(rd_env* env, int G, const rd_dreamer_weights* w, bool encoder, const rd_dreamer_conv_encoder* enc,
                 const int32_t* agent_of_env, const char* fn) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (encoder && !enc) return fail(env, RD_ERR_INVALID, "%s: null encoder", fn);
  if (encoder && !(env->cfg.obs_flags & RD_OBS_OCCUPANCY))
    return fail(env, RD_ERR_INVALID, "%s: the env does not produce lidar_occupancy (RD_OBS_OCCUPANCY)", fn);
  if (!encoder && (env->cfg.obs_flags & RD_OBS_LIDAR_F16))
    return fail(env, RD_ERR_INVALID, "the on-device policies read float32 scans: RD_OBS_LIDAR_F16 is set");
  const bool lidar_normalised = !encoder && (env->cfg.obs_flags & RD_OBS_LIDAR_NORM);
  const int rc = dreamer_init(env->dr, env->n, env->cfg.n_beams, lidar_normalised, G, w, enc, agent_of_env);
  if (rc) return fail(env, rc, "%s: %s", fn, env->dr.err.c_str());
  return ensure_rollout_actions(env);
}
// the four agent-step entry points: obs_dev is the scans or (encoder) the images; training reads eps_expl_dev as well
int step_dreamer(rd_env* env, const void* obs_dev, bool encoder, bool training, float* actions_dev, int noise,
                 const float* eps_stoch_dev, const float* eps_actor_dev, const float* eps_expl_dev, float* debug_dev,
                 void* stream, const char* fn) {
  if (!env || !obs_dev || !actions_dev) return fail(env, RD_ERR_INVALID, "null argument");
  if (int rc = dreamer_kind(env, encoder, fn)) return rc;
  if (noise < RD_NOISE_ZERO || noise > RD_NOISE_EXPLICIT) return fail(env, RD_ERR_INVALID, "bad noise mode %d", noise);
  if (noise == RD_NOISE_EXPLICIT && (!eps_stoch_dev || !eps_actor_dev || (training && !eps_expl_dev)))
    return fail(env, RD_ERR_INVALID, training ? "RD_NOISE_EXPLICIT needs eps_stoch_dev, eps_sample_dev and eps_expl_dev"
                                              : "RD_NOISE_EXPLICIT needs eps_stoch_dev and eps_actor_dev");
  return launch_dreamer(env, obs_dev, actions_dev, noise, eps_stoch_dev, eps_actor_dev, debug_dev, (cudaStream_t)stream,
                        training, eps_expl_dev);
}
// the checks every Dreamer rollout makes; *obs = what it feeds the agent: the scans, or an encoder agent's images
int dreamer_rollout_obs(rd_env* env, const rd_outputs* out, int noise, const void** obs) {
  if (!env->dr.ready) return fail(env, RD_ERR_STATE, "rd_policy_dreamer_init has not been called");
  if (!env->dr.depth) *obs = out->lidar_dev;
  else *obs = (env->cfg.obs_flags & RD_OBS_OCCUPANCY) ? out->occupancy_dev : nullptr;
  if (!*obs)
    return fail(env, RD_ERR_INVALID, env->dr.depth ? "the rollout needs out->occupancy_dev and an env that produces it (RD_OBS_OCCUPANCY)"
                                                   : "the rollout needs out->lidar_dev");
  if (noise != RD_NOISE_ZERO && noise != RD_NOISE_PHILOX)
    return fail(env, RD_ERR_INVALID, "a rollout draws its own noise (RD_NOISE_ZERO or RD_NOISE_PHILOX)");
  return RD_OK;
}
// rd_rollout_dreamer and _train
int rollout_dreamer(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, int noise, void* stream,
                    bool training) {
  if (!env || !out || n_steps < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  const void* obs = nullptr;
  if (int rc = dreamer_rollout_obs(env, out, noise, &obs)) return rc;
  if (!env->was_reset) return fail(env, RD_ERR_STATE, "Must reset environment.");
  float* act = actions_dev ? actions_dev : env->pol.d_actions;
  for (int k = 0; k < n_steps; ++k) {
    int rc = launch_dreamer(env, obs, act, noise, nullptr, nullptr, nullptr, (cudaStream_t)stream, training);
    if (rc) return rc;
    if ((rc = rd_step(env, act, out, stream))) return rc;
  }
  return RD_OK;
}
// rd_policy_dreamer_set_weights, _set_weights_occupancy (encoder: the latter, enc its image encoder) and
// _set_agent_weights (agent >= 0; -1: the single agent of the other two)
int set_dreamer_weights(rd_env* env, int agent, const rd_dreamer_weights* w, bool encoder, const rd_dreamer_conv_encoder* enc,
                        int on_device, void* stream, const char* fn) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (encoder && !enc) return fail(env, RD_ERR_INVALID, "%s: null encoder", fn);
  if (int rc = dreamer_kind(env, encoder, fn)) return rc;
  if (agent < 0 && env->dr.n_agents > 1)
    return fail(env, RD_ERR_INVALID, "%s: the policy has %d agents; use rd_policy_dreamer_set_agent_weights", fn, env->dr.n_agents);
  const int rc = dreamer_set_weights(env->dr, std::max(agent, 0), w, enc, on_device != 0, (cudaStream_t)stream);
  if (rc) return fail(env, rc, "%s: %s", fn, env->dr.err.c_str());
  env->launches += encoder ? 4 : 1;   // k_pack_weights, then k_pack_conv for conv2..conv4
  return RD_OK;
}
// the exploration state of agent `agent` (-1: the single agent of rd_policy_dreamer_get/set_exploration)
int dreamer_exploration(rd_env* env, int agent, rd_dreamer_exploration* x, bool set, const char* fn) {
  if (!env || !x) return fail(env, RD_ERR_INVALID, "null argument");
  if (!env->dr.ready) return fail(env, RD_ERR_STATE, "rd_policy_dreamer_init has not been called");
  if (agent < 0 && env->dr.n_agents > 1)
    return fail(env, RD_ERR_INVALID, "%s: the policy has %d agents; use the per-agent exploration calls", fn, env->dr.n_agents);
  if (agent >= env->dr.n_agents) return fail(env, RD_ERR_INVALID, "%s: agent %d is not in [0, n_agents)", fn, agent);
  rd_dreamer_exploration& e = env->dr.expl[std::max(agent, 0)];
  if (!set) { *x = e; return RD_OK; }
  if (!(x->amount >= 0.0) || !(x->decay >= 0.0) || !(x->min_amount >= 0.0) || x->env_steps < 0)
    return fail(env, RD_ERR_INVALID, "exploration: amount, decay, min_amount and env_steps must be >= 0");
  e = *x;
  return RD_OK;
}
}  // namespace

RD_API int rd_policy_dreamer_init(rd_env* env, const rd_dreamer_weights* w) {
  return init_dreamer(env, 1, w, false, nullptr, nullptr, "rd_policy_dreamer_init");
}

RD_API int rd_policy_dreamer(rd_env* env, const float* lidar_dev, float* actions_dev, int noise, const float* eps_stoch_dev,
                             const float* eps_actor_dev, float* debug_dev, void* stream) {
  return step_dreamer(env, lidar_dev, false, false, actions_dev, noise, eps_stoch_dev, eps_actor_dev, nullptr, debug_dev,
                      stream, "rd_policy_dreamer");
}

RD_API int rd_policy_dreamer_get_state(rd_env* env, float* stoch_dev, float* deter_dev, float* action_dev, void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (!env->dr.ready) return fail(env, RD_ERR_STATE, "rd_policy_dreamer_init has not been called");
  const int rc = dreamer_state_io(env->dr, stoch_dev, deter_dev, action_dev, 0, (cudaStream_t)stream);
  if (rc) return fail(env, rc, "rd_policy_dreamer_get_state: %s", env->dr.err.c_str());
  return RD_OK;
}

RD_API int rd_policy_dreamer_set_state(rd_env* env, const float* stoch_dev, const float* deter_dev, const float* action_dev,
                                       void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (!env->dr.ready) return fail(env, RD_ERR_STATE, "rd_policy_dreamer_init has not been called");
  const int rc = dreamer_state_io(env->dr, const_cast<float*>(stoch_dev), const_cast<float*>(deter_dev),
                                  const_cast<float*>(action_dev), 1, (cudaStream_t)stream);
  if (rc) return fail(env, rc, "rd_policy_dreamer_set_state: %s", env->dr.err.c_str());
  return RD_OK;
}

RD_API int rd_rollout_dreamer(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, int noise, void* stream) {
  return rollout_dreamer(env, n_steps, out, actions_dev, noise, stream, false);
}

RD_API int rd_policy_dreamer_train(rd_env* env, const float* lidar_dev, float* actions_dev, int noise, const float* eps_stoch_dev,
                                   const float* eps_sample_dev, const float* eps_expl_dev, float* debug_dev, void* stream) {
  return step_dreamer(env, lidar_dev, false, true, actions_dev, noise, eps_stoch_dev, eps_sample_dev, eps_expl_dev, debug_dev,
                      stream, "rd_policy_dreamer_train");
}

RD_API int rd_rollout_dreamer_train(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, int noise, void* stream) {
  return rollout_dreamer(env, n_steps, out, actions_dev, noise, stream, true);
}

RD_API int rd_policy_dreamer_set_exploration(rd_env* env, const rd_dreamer_exploration* x) {
  return dreamer_exploration(env, -1, const_cast<rd_dreamer_exploration*>(x), true, "rd_policy_dreamer_set_exploration");
}

RD_API int rd_policy_dreamer_get_exploration(rd_env* env, rd_dreamer_exploration* x) {
  return dreamer_exploration(env, -1, x, false, "rd_policy_dreamer_get_exploration");
}

RD_API int rd_policy_dreamer_set_weights(rd_env* env, const rd_dreamer_weights* w, int on_device, void* stream) {
  return set_dreamer_weights(env, -1, w, false, nullptr, on_device, stream, "rd_policy_dreamer_set_weights");
}

RD_API int rd_policy_dreamer_init_occupancy(rd_env* env, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc) {
  return init_dreamer(env, 1, w, true, enc, nullptr, "rd_policy_dreamer_init_occupancy");
}

RD_API int rd_policy_dreamer_init_agents(rd_env* env, int32_t n_agents, const rd_dreamer_weights* w,
                                         const rd_dreamer_conv_encoder* enc, const int32_t* agent_of_env_host) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (!w || !agent_of_env_host) return fail(env, RD_ERR_INVALID, "rd_policy_dreamer_init_agents: null argument");
  return init_dreamer(env, n_agents, w, enc != nullptr, enc, agent_of_env_host, "rd_policy_dreamer_init_agents");
}

RD_API int rd_policy_dreamer_set_agent_weights(rd_env* env, int32_t agent, const rd_dreamer_weights* w,
                                               const rd_dreamer_conv_encoder* enc, int on_device, void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (agent < 0) return fail(env, RD_ERR_INVALID, "rd_policy_dreamer_set_agent_weights: agent %d is not in [0, n_agents)", agent);
  return set_dreamer_weights(env, agent, w, enc != nullptr, enc, on_device, stream, "rd_policy_dreamer_set_agent_weights");
}

RD_API int rd_policy_dreamer_set_agent_exploration(rd_env* env, int32_t agent, const rd_dreamer_exploration* x) {
  if (agent < 0) return fail(env, RD_ERR_INVALID, "rd_policy_dreamer_set_agent_exploration: agent %d is not in [0, n_agents)", agent);
  return dreamer_exploration(env, agent, const_cast<rd_dreamer_exploration*>(x), true, "rd_policy_dreamer_set_agent_exploration");
}

RD_API int rd_policy_dreamer_get_agent_exploration(rd_env* env, int32_t agent, rd_dreamer_exploration* x) {
  if (agent < 0) return fail(env, RD_ERR_INVALID, "rd_policy_dreamer_get_agent_exploration: agent %d is not in [0, n_agents)", agent);
  return dreamer_exploration(env, agent, x, false, "rd_policy_dreamer_get_agent_exploration");
}

RD_API int rd_policy_dreamer_occupancy(rd_env* env, const uint8_t* occupancy_dev, float* actions_dev, int noise,
                                       const float* eps_stoch_dev, const float* eps_actor_dev, float* debug_dev, void* stream) {
  return step_dreamer(env, occupancy_dev, true, false, actions_dev, noise, eps_stoch_dev, eps_actor_dev, nullptr, debug_dev,
                      stream, "rd_policy_dreamer_occupancy");
}

RD_API int rd_policy_dreamer_occupancy_train(rd_env* env, const uint8_t* occupancy_dev, float* actions_dev, int noise,
                                             const float* eps_stoch_dev, const float* eps_sample_dev, const float* eps_expl_dev,
                                             float* debug_dev, void* stream) {
  return step_dreamer(env, occupancy_dev, true, true, actions_dev, noise, eps_stoch_dev, eps_sample_dev, eps_expl_dev,
                      debug_dev, stream, "rd_policy_dreamer_occupancy_train");
}

RD_API int rd_policy_dreamer_set_weights_occupancy(rd_env* env, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc,
                                                   int on_device, void* stream) {
  return set_dreamer_weights(env, -1, w, true, enc, on_device, stream, "rd_policy_dreamer_set_weights_occupancy");
}

RD_API int rd_dreamer_encode_occupancy(rd_env* env, const uint8_t* occupancy_dev, float* embed_dev, void* stream) {
  if (!env || !occupancy_dev || !embed_dev) return fail(env, RD_ERR_INVALID, "null argument");
  if (int rc = dreamer_kind(env, true, "rd_dreamer_encode_occupancy")) return rc;
  DreamerPolicy& d = env->dr;
  cudaStream_t s = (cudaStream_t)stream;
  int launched = 0;
  int rc = dreamer_encode(d, occupancy_dev, s, &launched);
  if (!rc) {   // embed = hi + lo: the latent copy kernel over [n][embed] rows
    const size_t total = (size_t)d.n * d.embed;
    k_latent_copy<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(d.lidar.p[0], d.lidar.p[1], d.embed, 0, d.embed, embed_dev, d.n, 0,
                                                                  d.row_of_env);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { rc = RD_ERR_CUDA; d.err = std::string("k_latent_copy: ") + cudaGetErrorString(e); }
    ++launched;
  }
  env->launches += launched;
  if (rc) return fail(env, rc, "rd_dreamer_encode_occupancy: %s", d.err.c_str());
  return RD_OK;
}

RD_API int rd_lidar_cast(rd_env* env, const double* poses_dev, const int32_t* map_ids_host, int n, float* ranges_dev,
                         void* stream) {
  if (!env || n < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  if (n == 0) return RD_OK;  // empty batch: nothing to do (pointers may be null)
  if (!poses_dev || !ranges_dev) return fail(env, RD_ERR_INVALID, "null pointer");
  if (env->cfg.agents_per_world > 1 && n % env->cfg.agents_per_world != 0)   // worlds = consecutive poses: whole worlds only
    return fail(env, RD_ERR_INVALID, "rd_lidar_cast: %d poses are not whole worlds of %d cars", n, env->cfg.agents_per_world);
  if (env->cfg.agents_per_world > 1 && map_ids_host)
    for (int e = 0; e < n; ++e)
      if (map_ids_host[e] != map_ids_host[e - e % env->cfg.agents_per_world])
        return fail(env, RD_ERR_INVALID, "rd_lidar_cast: pose %d: the cars of one world must share a map", e);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = sync_maps(env);
  if (rc) return rc;
  if ((rc = ensure_stage(env, n))) return rc;
  int runs[RD_MAX_MAPS][2];
  if ((rc = stage_runs(env, map_ids_host, n, runs, s))) return rc;
  k_origin_from_poses<<<(n + 127) / 128, 128, 0, s>>>(env->d_maps, map_ids_host ? env->d_stage_ids : nullptr, poses_dev, n,
                                                     env->cfg.lidar_offset, env->d_stage_recs);
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  for (int mid = 0; mid < RD_MAX_MAPS; ++mid) {
    if (runs[mid][1] == 0) continue;
    const size_t first = (size_t)runs[mid][0];
    rc = launch_lidar(env, mid, env->d_stage_recs + first, nullptr, runs[mid][1], ranges_dev + first * env->cfg.n_beams, s);
    if (rc) return rc;
  }
  return RD_OK;
}

RD_API int rd_occupancy_obs(rd_env* env, const double* poses_dev, const int32_t* map_ids_host, int n, uint8_t* out_dev,
                            void* stream) {
  if (!env || n < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  if (n == 0) return RD_OK;
  if (!poses_dev || !out_dev) return fail(env, RD_ERR_INVALID, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = sync_maps(env);
  if (rc) return rc;
  if ((rc = ensure_stage(env, n))) return rc;
  int runs[RD_MAX_MAPS][2];
  if ((rc = stage_runs(env, map_ids_host, n, runs, s))) return rc;
  for (int mid = 0; mid < RD_MAX_MAPS; ++mid) {
    if (runs[mid][1] == 0) continue;
    const size_t first = (size_t)runs[mid][0];
    rc = launch_occupancy(env, mid, nullptr, poses_dev + 3 * first, nullptr, runs[mid][1], out_dev + first * 4096, s);
    if (rc) return rc;
  }
  return RD_OK;
}

RD_API int rd_dynamics(rd_env* env, double* state_dev, const double* commands_dev, int n, int n_ticks, void* stream) {
  if (!env || n < 0 || n_ticks < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  if (n == 0) return RD_OK;
  if (!state_dev || !commands_dev) return fail(env, RD_ERR_INVALID, "null pointer");
  k_dynamics<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(env->vk, env->voff, env->d_vk, env->d_voff, state_dev, commands_dev, n, n_ticks);
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}

RD_API int rd_reward_done(rd_env* env, const double* kin_dev, const double* steering_dev, const int32_t* map_ids_host, int n,
                          double* book_f64_dev, int32_t* book_i32_dev, double* reward_dev, uint8_t* done_dev, void* stream) {
  if (!env || n < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  if (n == 0) return RD_OK;
  if (!kin_dev || !book_f64_dev || !book_i32_dev || !reward_dev || !done_dev) return fail(env, RD_ERR_INVALID, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = sync_maps(env);
  if (rc) return rc;
  if ((rc = ensure_stage(env, n))) return rc;
  int runs[RD_MAX_MAPS][2];
  if ((rc = stage_runs(env, map_ids_host, n, runs, s))) return rc;
  k_reward_done<<<(n + 127) / 128, 128, 0, s>>>(env->cfg, env->d_maps, map_ids_host ? env->d_stage_ids : nullptr, kin_dev,
                                               steering_dev, n, book_f64_dev, book_i32_dev, reward_dev, done_dev);
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}

RD_API int rd_get_state(rd_env* env, double* f64_dev, int32_t* i32_dev, void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)env->n;
  (void)n;
  if (f64_dev || i32_dev) {
    k_state_export<<<(env->n + 127) / 128, 128, 0, s>>>(step_params(env).S, f64_dev, i32_dev);
    env->launches++;
    CUDA_TRY(env, cudaGetLastError());
  }
  return RD_OK;
}

RD_API int rd_set_state(rd_env* env, const double* f64_dev, const int32_t* i32_dev, void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  if (!env->assigned) return fail(env, RD_ERR_STATE, "rd_assign_maps has not been called");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)env->n;
  (void)n;
  if (f64_dev || i32_dev) {
    // everything but the map column (owned by rd_assign_maps: the env grouping depends on it); the n-step ring is not
    // part of the state layout and restarts from the restored lap + progress
    k_state_import<<<(env->n + 127) / 128, 128, 0, s>>>(step_params(env).S, f64_dev, i32_dev, env->d_hist, env->cfg.n_step_progress);
    env->launches++;
    CUDA_TRY(env, cudaGetLastError());
  }
  env->was_reset = true;
  return RD_OK;
}

RD_API int rd_read_stats(rd_env* env, rd_stats* out_host, int reset, void* stream) {
  if (!env || !out_host) return fail(env, RD_ERR_INVALID, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  double h[RD_NSTAT];
  CUDA_TRY(env, cudaMemcpyAsync(h, env->d_stats, sizeof(h), cudaMemcpyDeviceToHost, s));
  if (reset) CUDA_TRY(env, cudaMemsetAsync(env->d_stats, 0, sizeof(h), s));
  CUDA_TRY(env, cudaStreamSynchronize(s));
  out_host->episodes = h[0]; out_host->return_sum = h[1]; out_host->progress_sum = h[2]; out_host->length_sum = h[3];
  out_host->collisions = h[4]; out_host->laps_completed = h[5]; out_host->env_steps = h[6]; out_host->timeouts = h[7];
  out_host->max_progress_sum = h[8];
  return RD_OK;
}

RD_API int rd_enable_timing(rd_env* env, int enable) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  env->timing = enable != 0;
  return RD_OK;
}

RD_API int rd_read_timing(rd_env* env, rd_timing* out_host, int reset) {
  if (!env || !out_host) return fail(env, RD_ERR_INVALID, "null argument");
  for (auto& t : env->timed) {
    CUDA_TRY(env, cudaEventSynchronize(t.b));
    float ms = 0.f;
    CUDA_TRY(env, cudaEventElapsedTime(&ms, t.a, t.b));
    switch (t.kind) {
      case T_STEP: env->acc.step_ms += ms; env->acc.step_launches++; break;
      case T_LIDAR: env->acc.lidar_ms += ms; env->acc.lidar_launches++; break;
      case T_OCC: env->acc.occupancy_ms += ms; env->acc.occupancy_launches++; break;
      case T_POLICY: env->acc.policy_ms += ms; env->acc.policy_launches++; break;
      default: env->acc.reset_ms += ms; env->acc.reset_launches++; break;
    }
    env->event_pool.push_back(t.a);
    env->event_pool.push_back(t.b);
  }
  env->timed.clear();
  *out_host = env->acc;
  if (reset) env->acc = rd_timing{};
  return RD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// device-resident episode store (csrc/rd_store.cuh)
namespace {
// Longest episode the config allows, in agent steps (-1: unbounded): TimeLimit in agent steps, the gym TimeLimit in
// ticks, and the tasks' time > time_limit (time advances by dt per tick, so that tick is at most floor(time_limit / dt)
// + 2 ticks away even with the rounding of the accumulated time).  A world ends with its first car.
int64_t store_max_steps(const rd_config& c) {
  const int64_t R = c.action_repeat;
  int64_t best = -1;
  auto take = [&](int64_t v) { if (best < 0 || v < best) best = v; };
  if (c.time_limit_steps > 0) take(c.time_limit_steps);
  if (c.time_limit_ticks > 0) take((c.time_limit_ticks + R - 1) / R);
  bool timed = false;   // max_speed has no time limit of its own [REF baselines/racing/environment/tasks.py:6-18]
  if (c.agents_per_world > 1) {
    for (int a = 0; a < c.agents_per_world; ++a) timed = timed || c.agent_task[a] != RD_TASK_MAX_SPEED;
  } else {
    timed = c.task != RD_TASK_MAX_SPEED;
  }
  if (timed && c.time_limit >= 0.0 && c.time_limit / c.dt < 1.0e15) {
    const double ticks = std::floor(c.time_limit / c.dt) + 2.0;
    take((int64_t)std::ceil(ticks / (double)R));
  }
  return best;
}

StoreSrc store_src(const rd_outputs* o, const float* actions) {
  StoreSrc r{};
  r.lidar = o->lidar_dev; r.occ = o->occupancy_dev; r.pose = o->pose_dev; r.vel = o->velocity_dev; r.speed = o->speed_dev;
  r.reward = o->reward_dev; r.done = o->done_dev; r.progress = o->progress_dev; r.lap = o->lap_dev; r.time = o->time_dev;
  r.actions = actions;
  return r;
}

int store_check_out(rd_env* env, const rd_outputs* o) {
  const auto& d = env->st.d;
  if (!o || !o->pose_dev || !o->velocity_dev || !o->speed_dev || !o->reward_dev || !o->done_dev || !o->progress_dev ||
      !o->lap_dev || !o->time_dev || (d.rows[SK_LIDAR] && !o->lidar_dev) || (d.rows[SK_OCC] && !o->occupancy_dev))
    return fail(env, RD_ERR_INVALID, "the episode store records pose, velocity, speed, reward, done, progress, lap, time "
                                     "and the stored observations: an output pointer is NULL");
  return RD_OK;
}

int store_mode(const rd_env* env) {
  return env->st.sc.reset_mode < 0 ? env->cfg.reset_mode : env->st.sc.reset_mode;
}

// ids of the held episodes of at least min_len rows, in commit order -> st.d_elig / st.d_n_elig (cached until the
// store changes)
int store_compact(rd_env* env, int min_len, cudaStream_t s) {
  auto& st = env->st;
  if (st.elig_epoch == st.epoch && st.elig_min == min_len) return RD_OK;
  StoreIdIter it(thrust::counting_iterator<int64_t>(0), StoreIdOf{st.d.next_id, st.d.M, st.d.Mi, st.d.imp_next});
  size_t bytes = st.cub_bytes;
  CUDA_TRY(env, cub::DeviceSelect::If(st.d_cub, bytes, it, st.d_elig, st.d_n_elig, (int)(st.d.M + st.d.Mi),
                                      StoreEligible{st.d, min_len}, s));
  env->launches++;
  st.elig_epoch = st.epoch;
  st.elig_min = min_len;
  return RD_OK;
}

// (id, env, rows) of every held episode, imported ones (n_imp of them) first; synchronises s
int store_held(rd_env* env, cudaStream_t s, std::vector<int64_t>& eps, int& n_imp) {
  auto& st = env->st;
  int rc = store_compact(env, 1, s);
  if (rc) return rc;
  int held = 0;
  CUDA_TRY(env, cudaMemcpyAsync(&held, st.d_n_elig, sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(env, cudaStreamSynchronize(s));
  eps.assign(3 * (size_t)held, 0);
  if (held > 0) {
    k_store_export<<<(held + 127) / 128, 128, 0, s>>>(st.d, st.d_elig, held, st.d_export);
    env->launches++;
    CUDA_TRY(env, cudaGetLastError());
    CUDA_TRY(env, cudaMemcpyAsync(eps.data(), st.d_export, sizeof(int64_t) * eps.size(), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(env, cudaStreamSynchronize(s));
  }
  n_imp = 0;
  while (n_imp < held && eps[3 * (size_t)n_imp] >= RD_STORE_IMPORTED_ID0) n_imp++;
  return RD_OK;
}

int store_record(rd_env* env, const rd_outputs* out, const float* actions, int reset_rows, cudaStream_t s) {
  k_store_record<<<env->n, 128, 0, s>>>(env->st.d, store_src(out, actions), reset_rows);
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}

int store_step(rd_env* env, const float* actions_dev, const rd_outputs* out, cudaStream_t s) {
  auto& st = env->st;
  int rc = rd_step(env, actions_dev, out, s);
  if (rc) return rc;
  if ((rc = store_record(env, out, actions_dev, 0, s))) return rc;
  k_store_commit<<<1, RD_COMMIT_THREADS, 0, s>>>(st.d, out->done_dev);
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  // reset of the committed envs; the others are marked frozen so that the observation kernels skip them, and reward /
  // done keep the finished step's values (what EpisodeRecorder.step returns)
  rd_outputs keep = *out;
  keep.reward_dev = nullptr;
  keep.done_dev = nullptr;
  {
    ScopedTiming tm(env, s, T_RESET);
    k_reset<<<(env->n + 127) / 128, 128, 0, s>>>(step_params(env), out_ptrs(&keep), st.d.fin, store_mode(env), 1);
  }
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  if ((rc = observe(env, &keep, s, 0, -1, nullptr, true))) return rc;
  if ((rc = store_record(env, out, actions_dev, 1, s))) return rc;
  st.epoch++;
  return RD_OK;
}
}  // namespace

RD_API int rd_store_init(rd_env* env, const rd_store_config* sc) {
  if (!env || !sc) return fail(env, RD_ERR_INVALID, "null argument");
  const rd_config& c = env->cfg;
  if (c.auto_reset)
    return fail(env, RD_ERR_INVALID, "the episode store needs auto_reset = 0: it records the terminal observation, then "
                                     "resets the finished envs itself");
  if (sc->precision != 32 && sc->precision != 16) return fail(env, RD_ERR_INVALID, "precision %d: expected 32 or 16", sc->precision);
  if (sc->keep_obs & ~31) return fail(env, RD_ERR_INVALID, "keep_obs 0x%x: unknown bits", sc->keep_obs);
  if ((sc->keep_obs & RD_STORE_OCCUPANCY) && !(c.obs_flags & RD_OBS_OCCUPANCY))
    return fail(env, RD_ERR_INVALID, "keep_obs has lidar_occupancy but the env does not produce it (RD_OBS_OCCUPANCY)");
  if (sc->reset_mode < -1 || sc->reset_mode > RD_RESET_RANDOM_BALL) return fail(env, RD_ERR_INVALID, "bad reset mode %d", sc->reset_mode);
  const int64_t max_steps = store_max_steps(c);
  if (max_steps < 0)
    return fail(env, RD_ERR_INVALID, "the config bounds no episode length (time_limit_steps, time_limit_ticks or a timed task): "
                                     "a ring could overwrite the episode in progress");
  if ((int64_t)sc->capacity_rows < max_steps + 1)
    return fail(env, RD_ERR_INVALID, "capacity_rows %d: episodes of this config reach %lld steps, so at least %lld rows are needed",
                sc->capacity_rows, (long long)max_steps, (long long)(max_steps + 1));
  const int64_t n = env->n, cap = sc->capacity_rows;
  const int64_t M = n * (cap + 2);
  if (M >= INT32_MAX) return fail(env, RD_ERR_INVALID, "n_envs x (capacity_rows + 2) = %lld exceeds the episode table's 2^31 slots", (long long)M);
  store_free(env->st);
  auto& st = env->st;
  st.sc = *sc;
  st.max_steps = max_steps;
  StoreDev& d = st.d;
  d.cap = (int)cap; d.n = (int)n; d.nb = c.n_beams; d.A = c.agents_per_world > 1 ? c.agents_per_world : 1; d.M = M;
  d.half = sc->precision == 16 ? 1 : 0;
  d.lidar_in_half = (c.obs_flags & RD_OBS_LIDAR_F16) ? 1 : 0;
  const int fe = d.half ? 2 : 4;
  const int rb[SK_N] = {c.n_beams * fe, 6 * fe, 6 * fe, fe, RD_OCC_OUT * RD_OCC_OUT, 2 * fe, fe, fe, fe, fe};
  const bool keep[SK_N] = {(sc->keep_obs & RD_STORE_LIDAR) != 0, (sc->keep_obs & RD_STORE_POSE) != 0,
                           (sc->keep_obs & RD_STORE_VELOCITY) != 0, (sc->keep_obs & RD_STORE_SPEED) != 0,
                           (sc->keep_obs & RD_STORE_OCCUPANCY) != 0, true, true, true, true, true};
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
  for (int k = 0; k < SK_N; ++k) {
    d.rb[k] = rb[k];
    if (keep[k]) alloc((void**)&d.rows[k], (size_t)n * (size_t)cap * (size_t)rb[k]);
  }
  alloc((void**)&d.head, sizeof(int64_t) * n);
  alloc((void**)&d.ep_start, sizeof(int64_t) * n);
  alloc((void**)&d.table, sizeof(StoreEp) * M);
  alloc((void**)&d.next_id, sizeof(int64_t));
  alloc((void**)&d.fin, (size_t)n);
  alloc((void**)&st.d_invalid, sizeof(unsigned long long));
  alloc((void**)&st.d_elig, sizeof(int64_t) * M);
  alloc((void**)&st.d_n_elig, sizeof(int));
  alloc((void**)&st.d_export, sizeof(int64_t) * 3 * M);
  if (e == cudaSuccess) e = cudaMemset(d.head, 0, sizeof(int64_t) * n);
  if (e == cudaSuccess) e = cudaMemset(d.ep_start, 0, sizeof(int64_t) * n);
  if (e == cudaSuccess) e = cudaMemset(d.table, 0xff, sizeof(StoreEp) * M);   // id -1: empty
  if (e == cudaSuccess) e = cudaMemset(d.next_id, 0, sizeof(int64_t));
  if (e == cudaSuccess) e = cudaMemset(d.fin, 0, (size_t)n);
  if (e == cudaSuccess) e = cudaMemset(st.d_invalid, 0, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemset(st.d_n_elig, 0, sizeof(int));
  if (e == cudaSuccess) {
    StoreIdIter it(thrust::counting_iterator<int64_t>(0), StoreIdOf{d.next_id, M, 0, 0});
    e = cub::DeviceSelect::If(nullptr, st.cub_bytes, it, st.d_elig, st.d_n_elig, (int)M, StoreEligible{d, 1});
  }
  alloc(&st.d_cub, std::max<size_t>(st.cub_bytes, 16));
  if (e != cudaSuccess) {
    cudaGetLastError();
    store_free(env->st);
    return fail(env, e == cudaErrorMemoryAllocation ? RD_ERR_NOMEM : RD_ERR_CUDA, "episode store allocation: %s", cudaGetErrorString(e));
  }
  st.ready = true;
  return RD_OK;
}

RD_API int rd_store_reset(rd_env* env, const rd_outputs* out, void* stream) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  auto& st = env->st;
  if (!st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  int rc = store_check_out(env, out);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = rd_reset(env, nullptr, store_mode(env), out, stream))) return rc;
  CUDA_TRY(env, cudaMemsetAsync(st.d.fin, 1, (size_t)env->n, s));
  if ((rc = store_record(env, out, nullptr, 1, s))) return rc;
  st.started = true;
  st.epoch++;
  return RD_OK;
}

RD_API int rd_store_step(rd_env* env, const float* actions_dev, const rd_outputs* out, void* stream) {
  if (!env || !actions_dev) return fail(env, RD_ERR_INVALID, "null argument");
  if (!env->st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  if (!env->st.started) return fail(env, RD_ERR_STATE, "rd_store_reset has not been called");
  int rc = store_check_out(env, out);
  if (rc) return rc;
  return store_step(env, actions_dev, out, (cudaStream_t)stream);
}

RD_API int rd_rollout_store(rd_env* env, int policy, int n_steps, const rd_outputs* out, float* actions_dev, int noise,
                            void* stream) {
  if (!env || n_steps < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  if (!env->st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  if (!env->st.started) return fail(env, RD_ERR_STATE, "rd_store_reset has not been called");
  int rc = store_check_out(env, out);
  if (rc) return rc;
  const void* dr_obs = nullptr;
  if (policy == RD_STORE_POLICY_GAP_FOLLOWER) {
    if (!out->lidar_dev) return fail(env, RD_ERR_INVALID, "the rollout needs out->lidar_dev");
    if (!env->pol.ready) return fail(env, RD_ERR_STATE, "rd_policy_gap_follower_init has not been called");
  } else if (policy == RD_STORE_POLICY_DREAMER || policy == RD_STORE_POLICY_DREAMER_TRAIN) {
    if ((rc = dreamer_rollout_obs(env, out, noise, &dr_obs))) return rc;
  } else {
    return fail(env, RD_ERR_INVALID, "bad policy %d", policy);
  }
  cudaStream_t s = (cudaStream_t)stream;
  float* act = actions_dev ? actions_dev : env->pol.d_actions;
  for (int k = 0; k < n_steps; ++k) {
    rc = policy == RD_STORE_POLICY_GAP_FOLLOWER ? launch_gap_follower(env, out->lidar_dev, nullptr, act, nullptr, s)
                                                : launch_dreamer(env, dr_obs, act, noise, nullptr, nullptr, nullptr, s,
                                                                 policy == RD_STORE_POLICY_DREAMER_TRAIN);
    if (rc) return rc;
    if ((rc = store_step(env, act, out, s))) return rc;
  }
  return RD_OK;
}

RD_API int rd_store_sample(rd_env* env, int batch, int length, int balance, const int64_t* ids_dev, const int32_t* starts_dev,
                           const rd_store_batch* out, void* stream) {
  if (!env || !out) return fail(env, RD_ERR_INVALID, "null argument");
  auto& st = env->st;
  if (!st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  if (batch < 1 || length < 1 || (int64_t)batch * length >= INT32_MAX)
    return fail(env, RD_ERR_INVALID, "batch %d x length %d: both must be positive and the product below 2^31", batch, length);
  if (ids_dev && !starts_dev) return fail(env, RD_ERR_INVALID, "explicit indices need both ids_dev and starts_dev");
  if (ids_dev) {   // k_store_gather reads the requests of entry b in every CTA of b while one of them writes its outputs
    auto overlap = [&](const void* a, size_t an, const void* b, size_t bn) {
      const uintptr_t a0 = (uintptr_t)a, b0 = (uintptr_t)b;
      return a && b && a0 < b0 + bn && b0 < a0 + an;
    };
    const size_t ni = sizeof(int64_t) * (size_t)batch, ns = sizeof(int32_t) * (size_t)batch;
    if (overlap(ids_dev, ni, out->episode_id_dev, ni) || overlap(ids_dev, ni, out->start_dev, ns) ||
        overlap(starts_dev, ns, out->episode_id_dev, ni) || overlap(starts_dev, ns, out->start_dev, ns))
      return fail(env, RD_ERR_INVALID, "the episode_id / start outputs overlap the explicit indices: pass separate buffers");
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (batch > st.req_cap) {   // scratch: requests [batch] and the id / start outputs [batch] when the caller gives none
    cudaFree(st.d_req_id); cudaFree(st.d_req_start);
    st.d_req_id = nullptr; st.d_req_start = nullptr; st.req_cap = 0;
    CUDA_TRY(env, cudaMalloc(&st.d_req_id, sizeof(int64_t) * 2 * (size_t)batch));
    CUDA_TRY(env, cudaMalloc(&st.d_req_start, sizeof(int32_t) * 2 * (size_t)batch));
    st.req_cap = batch;
  }
  const int64_t* rid = ids_dev;
  const int32_t* rstart = starts_dev;
  if (!ids_dev) {
    int rc = store_compact(env, length + 1, s);   // the reference skips episodes with total - length < 1
    if (rc) return rc;
    const uint64_t seed = st.sc.seed;
    k_store_draw<<<(batch + 127) / 128, 128, 0, s>>>(st.d, st.d_elig, st.d_n_elig, batch, length, balance ? 1 : 0,
                                                     (uint32_t)seed, (uint32_t)(seed >> 32) ^ RD_STREAM_STORE,
                                                     (uint32_t)st.draws, st.d_req_id, st.d_req_start);
    env->launches++;
    CUDA_TRY(env, cudaGetLastError());
    st.draws++;
    rid = st.d_req_id;
    rstart = st.d_req_start;
  }
  StoreOut o{};
  o.p[SK_LIDAR] = (unsigned char*)out->lidar_dev; o.p[SK_POSE] = (unsigned char*)out->pose_dev;
  o.p[SK_VELOCITY] = (unsigned char*)out->velocity_dev; o.p[SK_SPEED] = (unsigned char*)out->speed_dev;
  o.p[SK_OCC] = out->occupancy_dev; o.p[SK_ACTION] = (unsigned char*)out->action_dev;
  o.p[SK_REWARD] = (unsigned char*)out->reward_dev; o.p[SK_DISCOUNT] = (unsigned char*)out->discount_dev;
  o.p[SK_PROGRESS] = (unsigned char*)out->progress_dev; o.p[SK_TIME] = (unsigned char*)out->time_dev;
  o.id = out->episode_id_dev ? out->episode_id_dev : st.d_req_id + st.req_cap;
  o.start = out->start_dev ? out->start_dev : st.d_req_start + st.req_cap;
  k_store_gather<<<(unsigned)((int64_t)batch * length), 128, 0, s>>>(st.d, o, rid, rstart, length, ids_dev ? 1 : 0, st.d_invalid);
  env->launches++;
  CUDA_TRY(env, cudaGetLastError());
  return RD_OK;
}

RD_API int rd_store_info(rd_env* env, rd_store_summary* out_host, rd_store_episode* episodes_host, int64_t max_episodes,
                         void* stream) {
  if (!env || !out_host) return fail(env, RD_ERR_INVALID, "null argument");
  auto& st = env->st;
  if (!st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t committed = 0;
  unsigned long long invalid = 0;
  CUDA_TRY(env, cudaMemcpyAsync(&committed, st.d.next_id, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(env, cudaMemcpyAsync(&invalid, st.d_invalid, sizeof(invalid), cudaMemcpyDeviceToHost, s));
  std::vector<int64_t> all;
  int n_imp = 0;
  int rc = store_held(env, s, all, n_imp);
  if (rc) return rc;
  const int held = (int)(all.size() / 3) - n_imp;   // the recorded episodes follow the imported ones
  const int64_t* eps = all.data() + 3 * (size_t)n_imp;
  int64_t rows = 0;
  for (int i = 0; i < held; ++i) rows += eps[3 * (size_t)i + 2];
  out_host->committed = committed;
  out_host->held = held;
  out_host->held_rows = rows;
  out_host->evicted = committed - held;
  out_host->invalid_requests = (int64_t)invalid;
  out_host->draws = st.draws;
  out_host->capacity_rows = st.sc.capacity_rows;
  out_host->max_episode_steps = st.max_steps;
  if (episodes_host)
    for (int64_t i = 0; i < std::min<int64_t>(held, max_episodes); ++i) {
      episodes_host[i].id = eps[3 * i]; episodes_host[i].env = eps[3 * i + 1]; episodes_host[i].length = eps[3 * i + 2];
    }
  return RD_OK;
}

RD_API int rd_store_import_init(rd_env* env, int32_t import_capacity_rows) {
  if (!env) return fail(nullptr, RD_ERR_INVALID, "null handle");
  auto& st = env->st;
  if (!st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  if (import_capacity_rows < 1) return fail(env, RD_ERR_INVALID, "import_capacity_rows %d: expected at least 1", import_capacity_rows);
  const int64_t icap = import_capacity_rows, Mi = icap + 1;
  if (st.d.M + Mi >= INT32_MAX)
    return fail(env, RD_ERR_INVALID, "the recorded and imported episode tables (%lld + %lld slots) exceed 2^31",
                (long long)st.d.M, (long long)Mi);
  StoreDev& d = st.d;
  // the new buffers are allocated first, so that a failed allocation leaves the store as it was
  unsigned char* imp[SK_N] = {};
  StoreEp* itable = nullptr; int64_t* elig = nullptr; int64_t* xport = nullptr; void* cub = nullptr;
  size_t cub_bytes = 0;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
  for (int k = 0; k < SK_N; ++k)
    if (d.rows[k]) alloc((void**)&imp[k], (size_t)icap * (size_t)d.rb[k]);
  alloc((void**)&itable, sizeof(StoreEp) * Mi);
  alloc((void**)&elig, sizeof(int64_t) * (d.M + Mi));
  alloc((void**)&xport, sizeof(int64_t) * 3 * (d.M + Mi));
  if (e == cudaSuccess) e = cudaMemset(itable, 0xff, sizeof(StoreEp) * Mi);   // id -1: empty
  if (e == cudaSuccess) {
    StoreIdIter it(thrust::counting_iterator<int64_t>(0), StoreIdOf{d.next_id, d.M, Mi, 0});
    e = cub::DeviceSelect::If(nullptr, cub_bytes, it, elig, st.d_n_elig, (int)(d.M + Mi), StoreEligible{d, 1});
  }
  alloc(&cub, std::max<size_t>(cub_bytes, 16));
  if (e != cudaSuccess) {
    cudaGetLastError();
    for (int k = 0; k < SK_N; ++k) cudaFree(imp[k]);
    cudaFree(itable); cudaFree(elig); cudaFree(xport); cudaFree(cub);
    return fail(env, e == cudaErrorMemoryAllocation ? RD_ERR_NOMEM : RD_ERR_CUDA, "import arena allocation: %s", cudaGetErrorString(e));
  }
  for (int k = 0; k < SK_N; ++k) { cudaFree(d.imp[k]); d.imp[k] = imp[k]; }
  cudaFree(d.itable); cudaFree(st.d_elig); cudaFree(st.d_export); cudaFree(st.d_cub);
  d.itable = itable; st.d_elig = elig; st.d_export = xport; st.d_cub = cub; st.cub_bytes = cub_bytes;
  d.icap = (int)icap; d.Mi = Mi; d.imp_head = 0; d.imp_next = 0;
  st.epoch++;
  return RD_OK;
}

RD_API int rd_store_import(rd_env* env, int32_t n_episodes, const int32_t* lengths_host, const rd_store_import_rows* rows,
                           void* stream) {
  if (!env || (n_episodes > 0 && !lengths_host) || n_episodes < 0) return fail(env, RD_ERR_INVALID, "bad argument");
  auto& st = env->st;
  StoreDev& d = st.d;
  if (!st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  if (d.icap == 0) return fail(env, RD_ERR_STATE, "the store has no import arena (rd_store_import_init)");
  if (n_episodes == 0) return RD_OK;
  std::vector<int64_t> first((size_t)n_episodes);
  int64_t total = 0;
  for (int j = 0; j < n_episodes; ++j) {
    if (lengths_host[j] < 1 || lengths_host[j] > d.icap)
      return fail(env, RD_ERR_INVALID, "episode %d of the import has %d rows: expected 1 to import_capacity_rows = %d", j,
                  lengths_host[j], d.icap);
    first[(size_t)j] = total;
    total += lengths_host[j];
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (rows) {
    StoreStaged in{};
    const void* p[SK_N] = {rows->lidar_dev, rows->pose_dev, rows->velocity_dev, rows->speed_dev, rows->occupancy_dev,
                           rows->action_dev, rows->reward_dev, rows->discount_dev, rows->progress_dev, rows->time_dev};
    const int32_t ty[SK_N] = {rows->lidar_type, rows->pose_type, rows->velocity_type, rows->speed_type, rows->occupancy_type,
                              rows->action_type, rows->reward_type, rows->discount_type, rows->progress_type, rows->time_type};
    const int32_t ne[SK_N] = {d.nb, 6, 6, 1, RD_OCC_OUT * RD_OCC_OUT, 2, 1, 1, 1, 1};
    static const char* names[SK_N] = {"lidar", "pose", "velocity", "speed", "lidar_occupancy", "action", "reward",
                                      "discount", "progress", "time"};
    for (int k = 0; k < SK_N; ++k) {
      if (!d.imp[k]) continue;
      const bool ok_ty = k == SK_OCC ? ty[k] == RD_STORE_U8 : (ty[k] == RD_STORE_F16 || ty[k] == RD_STORE_F32 || ty[k] == RD_STORE_F64);
      if (!p[k] || !ok_ty) return fail(env, RD_ERR_INVALID, "import rows of '%s': missing or of element type %d", names[k], ty[k]);
      in.p[k] = (const unsigned char*)p[k];
      in.type[k] = ty[k];
      in.ne[k] = ne[k];
    }
    if (n_episodes > st.imp_meta_cap) {
      cudaFree(st.d_imp_len); cudaFree(st.d_imp_first);
      st.d_imp_len = nullptr; st.d_imp_first = nullptr; st.imp_meta_cap = 0;
      CUDA_TRY(env, cudaMalloc(&st.d_imp_len, sizeof(int32_t) * (size_t)n_episodes));
      CUDA_TRY(env, cudaMalloc(&st.d_imp_first, sizeof(int64_t) * (size_t)n_episodes));
      st.imp_meta_cap = n_episodes;
    }
    CUDA_TRY(env, cudaMemcpyAsync(st.d_imp_len, lengths_host, sizeof(int32_t) * (size_t)n_episodes, cudaMemcpyHostToDevice, s));
    CUDA_TRY(env, cudaMemcpyAsync(st.d_imp_first, first.data(), sizeof(int64_t) * (size_t)n_episodes, cudaMemcpyHostToDevice, s));
    const int64_t grid = std::min<int64_t>(total, d.icap);
    k_store_import<<<(unsigned)grid, 128, 0, s>>>(d, in, total, st.d_imp_len, st.d_imp_first, n_episodes);
    env->launches++;
    CUDA_TRY(env, cudaGetLastError());
  }
  d.imp_head += total;
  d.imp_next += n_episodes;
  st.epoch++;
  return RD_OK;
}

RD_API int rd_store_import_info(rd_env* env, rd_store_import_summary* out_host, rd_store_episode* episodes_host,
                                int64_t max_episodes, void* stream) {
  if (!env || !out_host) return fail(env, RD_ERR_INVALID, "null argument");
  auto& st = env->st;
  if (!st.ready) return fail(env, RD_ERR_STATE, "rd_store_init has not been called");
  std::vector<int64_t> eps;
  int n_imp = 0;
  int rc = store_held(env, (cudaStream_t)stream, eps, n_imp);
  if (rc) return rc;
  int64_t rows = 0;
  for (int i = 0; i < n_imp; ++i) rows += eps[3 * (size_t)i + 2];
  out_host->imported = st.d.imp_next;
  out_host->held = n_imp;
  out_host->held_rows = rows;
  out_host->evicted = st.d.imp_next - n_imp;
  out_host->capacity_rows = st.d.icap;
  if (episodes_host)
    for (int64_t i = 0; i < std::min<int64_t>(n_imp, max_episodes); ++i) {
      episodes_host[i].id = eps[3 * i]; episodes_host[i].env = eps[3 * i + 1]; episodes_host[i].length = eps[3 * i + 2];
    }
  return RD_OK;
}
