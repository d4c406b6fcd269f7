// rd_dynamics.cuh -- K2: action transform + single-track dynamics + progress/lap/collision + reward/done
// + TimeLimit + auto-reset, one thread per env (SURVEY.md §8 a1, a3, a4, a7-a10).
//
// Replaces, fused into one pass: ReduceActionSpace._normalize [REF dreamer/wrappers.py:129-134] (and the
// baselines clip [REF baselines/racing/environment/single_agent.py:55-56]), ActionRepeat.step
// [REF dreamer/wrappers.py:107-116], MultiAgentRaceEnv.step -> pybullet.stepSimulation + task reward/done
// (racecar_gym, not in tree; call site [REF dreamer/wrappers.py:63-64]), RaceCarWrapper's speed obs
// [REF dreamer/wrappers.py:66], TimeLimit.step [REF dreamer/wrappers.py:147-154] and, for the model-free chain, gym's
// TimeLimit inside ActionRepeat and NormalizeObservations [REF baselines/racing/experiments/acme/experiment.py:66-75].
//
// Env state is SoA of 16-byte groups (double2 pairs, one int4 + one int2 per env): every state access of a thread is a
// 128-bit load or store and a warp's request for one group is 512 contiguous bytes.  The vehicle model (rd_vehicle.cuh)
// is float64; everything that decides an integer (cell lookups, checkpoint index, reward bookkeeping) keeps the CPU
// oracle's operation order (the translation unit is compiled with -fmad=false), so flags, laps and termination are
// bit-exact against it.
#pragma once
#include "rd_common.cuh"
#include "rd_vehicle.cuh"
#include "rd_lidar.cuh"
#include "rd_policy.cuh"

// ---- env state ----
enum { RD_P_XY = 0, RD_P_SV, RD_P_YW, RD_P_ST, RD_P_PL, RD_P_RS, RD_P_MP, RD_NPAIR };   // (x,y) (steer,v) (yaw,yaw_rate)
static_assert(2 * RD_NPAIR >= RD_NF64, "pair layout covers rd_env.h's float64 fields"); // (slip,time) (progress,last)
struct StateRef {                                                                       // (return,start) (maxprog,-)
  double2* f2;   // [RD_NPAIR][n]
  int4* i4;      // [n] lap, checkpoint, flags, agent_step
  int2* i2;      // [n] episode, map
  int n;
};
__device__ __forceinline__ double2 rd_ldp(const StateRef& S, int pair, int e) { return S.f2[(size_t)pair * S.n + e]; }
__device__ __forceinline__ void rd_stp(const StateRef& S, int pair, int e, double a, double b) {
  S.f2[(size_t)pair * S.n + e] = make_double2(a, b);
}

struct StepParams {
  rd_config cfg;
  VehConst vk;      // vehicle constants (host-computed once per handle)
  VehAcc off;       // dynamic-regime coefficients at zero acceleration
  const VehConst* vk_g;   // the same two structs in global memory (the out-of-line general tick takes their address)
  const VehAcc* off_g;
  StateRef S;
  double* stats;    // [RD_NSTAT] accumulators (rd_stats order)
  OriginRec* recs;  // [n]
  const DevMap* maps;
  PolicyState pol;  // on-device controller state, cleared with the env (null pointers: no policy attached)
  double* hist;     // [n_step_progress][n] ring of lap + progress per sim tick (n_step_progress task), or null
  double norm_lo[3], norm_sc[3];   // RD_OBS_NORM_BASELINES: low and 1 / (high - low) of lidar / pose / velocity
  int norm;         // 1: pose and velocity outputs are normalised
  int n;
};
#define RD_NSTAT 9

struct OutPtrs {
  float* pose; float* velocity; float* speed; float* reward; uint8_t* done; float* progress; int32_t* lap;
  float* time; uint8_t* flags; uint8_t* occupancy; int32_t* rank; uint8_t* opponents; uint8_t* wrong_way;
  uint8_t* wall_collision;
};

__device__ __forceinline__ int rd_checkpoint_of(const rd_config& cfg, double p) {
  int c = (int)(p * (double)cfg.n_checkpoints);
  return c > cfg.n_checkpoints - 1 ? cfg.n_checkpoints - 1 : c;
}
__device__ __forceinline__ bool rd_progress_at(const DevMap& m, double x, double y, double& p) {
  int cx, cy;
  if (!rd_cell_of(m, x, y, cx, cy)) return false;
  if (!rd_drivable_at(m, cx, cy)) return false;
  p = rdv_div_by((double)__ldg(m.dist + (size_t)cy * m.w + cx), (double)m.dmax, m.inv_dmax);
  return true;
}

// Footprint + progress probe of one pose, split in two so that the loads of tick t are in flight while tick t+1 is
// integrated (k_step): rd_probe_issue computes the five cells (centre + the four body corners) and issues the five bit
// loads plus the centre's wavefront distance; rd_probe_finish turns them into (collision, inside, progress).
// Same results as the oracle's collides() + cell_of() + progress_at().
struct Probe {
  uint32_t w[5];     // bit-grid word of each point (0 when the point is outside the crop)
  uint32_t dval;     // wavefront distance of the centre cell
  int sh[5];         // bit index inside the word
  bool in0;          // centre inside the crop
  double c, s;       // cos / sin of the heading (reused for the observation record)
};
__device__ __forceinline__ void rd_probe_issue_cs(const rd_config& cfg, const DevMap& m, double x, double y, double c, double s, Probe& pr);
__device__ __forceinline__ void rd_probe_issue(const rd_config& cfg, const DevMap& m, double x, double y, double yaw, Probe& pr) {
  double c, s;
  rdv_sincos(yaw, s, c);
  rd_probe_issue_cs(cfg, m, x, y, c, s, pr);
}
// ... with the cosine / sine of the heading already known
__device__ __forceinline__ void rd_probe_issue_cs(const rd_config& cfg, const DevMap& m, double x, double y, double c, double s, Probe& pr) {
  pr.c = c; pr.s = s;
  const double hl = 0.5 * cfg.vehicle.body_length, hw = 0.5 * cfg.vehicle.body_width;
  const double ax = hl * c, ay = hl * s, bx = hw * s, by = hw * c;
  const double px[5] = {x, (x + ax) - bx, (x + ax) + bx, (x - ax) - bx, (x - ax) + bx};
  const double py[5] = {y, (y + ay) + by, (y + ay) - by, (y - ay) + by, (y - ay) - by};
  int cx0 = 0, cy0 = 0;
  // one range guard for the whole footprint instead of one per point: when the centre is within 1e8 cells of the map
  // origin every corner (a body length away) passes rd_cell_of's |.| < 1e9 test, so the unguarded conversion below is
  // the same arithmetic; anything else (far away, NaN) takes the guarded form
  const double uc = (x - m.ox) * m.inv_res, vc = (y - m.oy) * m.inv_res;
  const bool near = fabs(uc) < 1.0e8 && fabs(vc) < 1.0e8;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    int cx, cy;
    bool in;
    if (near) {
      cx = (int)floor((px[k] - m.ox) * m.inv_res) - m.col0;
      cy = (int)floor((py[k] - m.oy) * m.inv_res) - m.row0;
      in = (unsigned)cx < (unsigned)m.w && (unsigned)cy < (unsigned)m.h;
    } else {
      in = rd_cell_of(m, px[k], py[k], cx, cy);
    }
    pr.w[k] = in ? __ldg(m.bits + (size_t)cy * m.rw + (cx >> 5)) : 0u;
    pr.sh[k] = cx & 31;
    if (k == 0) { pr.in0 = in; cx0 = cx; cy0 = cy; }
  }
  pr.dval = pr.in0 ? (uint32_t)__ldg(m.dist + (size_t)cy0 * m.w + cx0) : 0u;
}
__device__ __forceinline__ void rd_probe_finish(const DevMap& m, const Probe& pr, bool& col, bool& inside, double& p) {
  uint32_t free_all = 1u;
#pragma unroll
  for (int k = 0; k < 5; ++k) free_all &= pr.w[k] >> pr.sh[k];
  col = !(free_all & 1u);
  inside = pr.in0;
  if ((pr.w[0] >> pr.sh[0]) & 1u) p = rdv_div_by((double)pr.dval, (double)m.dmax, m.inv_dmax);
}

// a7: checkpoint / lap / wrong-way state machine of one tick [NEW-SPEC, SURVEY.md §8-a7]
__device__ __forceinline__ void rd_lap_machine(const rd_config& cfg, double p, int& lap, int& cp, int& flags) {
  const int ncp = cfg.n_checkpoints;
  const int cn = rd_checkpoint_of(cfg, p);
  if (cn == cp + 1) { cp = cn; flags &= ~RD_F_WRONG_WAY; }
  else if (cp == ncp - 1 && cn == 0 && ncp > 1) { lap += 1; cp = 0; flags &= ~RD_F_WRONG_WAY; }
  else if (cn == cp - 1 || (cp == 0 && cn == ncp - 1 && ncp > 1)) { flags |= RD_F_WRONG_WAY; }
}
// a8: the tick's reward and the task's done.  `hit`: the task's collision (walls, or walls + other cars in worlds);
// `ref`: lap + progress the progress reward is measured from (the previous tick, or n ticks back for n_step_progress)
__device__ __forceinline__ double rd_task_reward(const rd_config& cfg, int task, bool hit, double cur, double ref,
                                                 double steer_cmd, double v, double slip, int lap, double time, bool& d) {
  if (task == RD_TASK_MAX_SPEED) {  // [REF baselines/racing/environment/tasks.py:6-18]
    d = false;
    return hit ? -1.0 : -exp(fabs(steer_cmd) - v * cos(slip));
  }
  // maximize_progress [REF dreamer/scenarios/max_progress/austria.yml:8-10]
  double delta = cur - ref;
  if (delta > 0.5) delta = delta - 1.0;
  if (delta < -0.5) delta = delta + 1.0;
  if (cfg.progress_abs) delta = fabs(delta);
  double r = cfg.frame_reward + cfg.progress_reward * delta;
  if (hit) r = r + cfg.collision_reward;
  d = (cfg.terminate_on_collision && hit) || (lap > cfg.laps) || (time > cfg.time_limit);
  return r;
}
// a4 [REF dreamer/wrappers.py:129-134; baselines single_agent.py:55-56]: numpy keeps (action+1)/2 of a float32 policy
// output in float32 and promotes to float64 at `* (high-low)` (float64 arrays).
__device__ __forceinline__ double rd_action(const rd_config& cfg, float af, int k) {
  if (cfg.clip_actions) af = af < -1.0f ? -1.0f : (af > 1.0f ? 1.0f : af);
  if (cfg.rescale_actions) {
    const float t = __fdiv_rn(__fadd_rn(af, 1.0f), 2.0f);
    return (double)t * (cfg.action_high[k] - cfg.action_low[k]) + cfg.action_low[k];
  }
  return (double)af;
}

// reset of one env: pose from the map's tables (grid slot or a Philox-sampled candidate); writes the whole state and
// returns the pose in q (all rates zero) [REF dreamer/wrappers.py:91-92 reset(mode=...); sampler itself is racecar_gym
// -> NEW-SPEC]
// ... the pose and its progress (reads only: the same (env, episode) always yields the same pose, so k_step_split looks
// it up ahead of time for every env)
__device__ __forceinline__ void rd_reset_pose(const StepParams& P, const DevMap& m, int e, int mode, uint32_t episode,
                                              double& x, double& y, double& yaw, double& p) {
  const rd_config& cfg = P.cfg;
  // multi-agent worlds: the cars of a world draw ONE anchor (counter = global id of the world's agent 0) and line up
  // along the ball_next chain (cfg.ball_spacing metres of track apart); 'grid' hands out the staggered start slots
  const int A = cfg.agents_per_world > 1 ? cfg.agents_per_world : 1;
  const int a = e % A;
  const uint64_t gid = (uint64_t)(cfg.env_id_offset + (e - a));
  if (mode == RD_RESET_GRID || m.n_reset <= 0) {
    const int slot = a < m.n_start ? a : m.n_start - 1;
    x = m.start[3 * slot]; y = m.start[3 * slot + 1]; yaw = m.start[3 * slot + 2];
  } else {
    uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), episode, 0u};
    philox4x32_10(c, (uint32_t)cfg.seed, (uint32_t)(cfg.seed >> 32) ^ RD_STREAM_RESET);
    uint32_t idx = __umulhi(c[0], (uint32_t)m.n_reset);
    for (int k = 0; k < a && m.ball_next; ++k) idx = (uint32_t)__ldg(m.ball_next + idx);
    x = m.reset[3 * idx]; y = m.reset[3 * idx + 1]; yaw = m.reset[3 * idx + 2];
    if (mode == RD_RESET_RANDOM_BIDIRECTIONAL && (c[1] & 1u)) yaw = yaw + 3.14159265358979323846;
  }
  p = 0.0;
  rd_progress_at(m, x, y, p);
}
// ... and the state it leaves behind
__device__ __forceinline__ void rd_reset_commit(const StepParams& P, int e, uint32_t episode, int map_id, double x, double y,
                                                double yaw, double p, double (&q)[7]) {
  const rd_config& cfg = P.cfg;
  const int n = P.n;
  const StateRef& S = P.S;
  rd_stp(S, RD_P_XY, e, x, y);
  rd_stp(S, RD_P_SV, e, 0.0, 0.0);
  rd_stp(S, RD_P_YW, e, yaw, 0.0);
  rd_stp(S, RD_P_ST, e, 0.0, 0.0);
  rd_stp(S, RD_P_PL, e, p, 1.0 + p);
  rd_stp(S, RD_P_RS, e, 0.0, 1.0 + p);
  rd_stp(S, RD_P_MP, e, -1.0, 0.0);
  S.i4[e] = make_int4(1, rd_checkpoint_of(cfg, p), 0, 0);
  S.i2[e] = make_int2((int)(episode + 1u), map_id);
  if (P.hist) for (int k = 0; k < cfg.n_step_progress; ++k) P.hist[(size_t)k * n + e] = 1.0 + p;
  if (P.pol.i32 || P.pol.dr_feat) rd_policy_clear(P.pol, n, e);
  q[0] = x; q[1] = y; q[2] = 0.0; q[3] = 0.0; q[4] = yaw; q[5] = 0.0; q[6] = 0.0;
}
__device__ __forceinline__ void rd_reset_one(const StepParams& P, const DevMap& m, int e, int mode, uint32_t episode,
                                             int map_id, double (&q)[7], double& p_out) {
  double x, y, yaw, p;
  rd_reset_pose(P, m, e, mode, episode, x, y, yaw, p);
  rd_reset_commit(P, e, episode, map_id, x, y, yaw, p, q);
  p_out = p;
}

// observation scalars + the origin record for the LiDAR / occupancy kernels, from the committed pose.
// have_cs: (c, s) = cos / sin of q[4] are already known (the last tick's footprint probe)
struct ObsVals {            // what one env's step hands to the observation kernels and to the caller
  OriginRec rec;
  float pose[6], vel[6], speed;
};
#define RD_OBS_WORDS 25     // 12 (record) + 6 + 6 + 1 32-bit words
__device__ __forceinline__ void rd_obs_compute(const StepParams& P, const DevMap& m, int e, int map_id, const double (&q)[7],
                                               uint32_t episode, uint32_t agent_step, int was_reset, bool have_cs, double c,
                                               double s, ObsVals& ov) {
  const double x = q[0], y = q[1], yaw = q[4], v = q[3], slip = q[6];
  if (!have_cs) rdv_sincos(yaw, s, c);
  OriginRec& rec = ov.rec;
  rd_make_origin_cs(m, x, y, c, s, P.cfg.lidar_offset, rec);
  rec.gid = (uint32_t)(P.cfg.env_id_offset + e);   // noise counter: the low 32 bits of the global env id
  rec.episode = episode;
  rec.step = agent_step;
  rec.was_reset = was_reset;
  rec.pad = map_id;
  const double two_pi = 6.283185307179586;
  const double wy = yaw - rint(yaw / two_pi) * two_pi;
  double ss, cs;
  if (fabs(slip) < 0.78) rdv_sincos_kernel(slip, ss, cs); else rdv_sincos(slip, ss, cs);
  const double vx = v * cs, vy = v * ss;
  const double yr = q[5];
  if (P.norm) {   // NormalizeObservations: (x - low) * scaler in float64, then float32 [REF baselines single_agent.py:92-99]
    const double pl = P.norm_lo[RD_NORM_POSE], psc = P.norm_sc[RD_NORM_POSE];
    const double vl = P.norm_lo[RD_NORM_VELOCITY], vsc = P.norm_sc[RD_NORM_VELOCITY];
    const float zp = (float)((0.0 - pl) * psc), zv = (float)((0.0 - vl) * vsc);
    ov.pose[0] = (float)((x - pl) * psc); ov.pose[1] = (float)((y - pl) * psc);
    ov.pose[2] = zp; ov.pose[3] = zp; ov.pose[4] = zp; ov.pose[5] = (float)((wy - pl) * psc);
    ov.vel[0] = (float)((vx - vl) * vsc); ov.vel[1] = (float)((vy - vl) * vsc);
    ov.vel[2] = zv; ov.vel[3] = zv; ov.vel[4] = zv; ov.vel[5] = (float)((yr - vl) * vsc);
  } else {
    ov.pose[0] = (float)x; ov.pose[1] = (float)y; ov.pose[2] = 0.f; ov.pose[3] = 0.f; ov.pose[4] = 0.f; ov.pose[5] = (float)wy;
    ov.vel[0] = (float)vx; ov.vel[1] = (float)vy; ov.vel[2] = 0.f; ov.vel[3] = 0.f; ov.vel[4] = 0.f; ov.vel[5] = (float)yr;
  }
  ov.speed = (float)sqrt(vx * vx + vy * vy);  // [REF dreamer/wrappers.py:66]
}
__device__ __forceinline__ void rd_obs_store(const StepParams& P, const OutPtrs& o, int e, const ObsVals& ov) {
  P.recs[e] = ov.rec;
  if (o.pose) {
    float2* p2 = reinterpret_cast<float2*>(o.pose + (size_t)e * 6);   // rows are 24 bytes: 8-byte aligned float2 stores
    p2[0] = make_float2(ov.pose[0], ov.pose[1]); p2[1] = make_float2(ov.pose[2], ov.pose[3]); p2[2] = make_float2(ov.pose[4], ov.pose[5]);
  }
  if (o.velocity) {
    float2* q2 = reinterpret_cast<float2*>(o.velocity + (size_t)e * 6);
    q2[0] = make_float2(ov.vel[0], ov.vel[1]); q2[1] = make_float2(ov.vel[2], ov.vel[3]); q2[2] = make_float2(ov.vel[4], ov.vel[5]);
  }
  if (o.speed) o.speed[e] = ov.speed;
}
__device__ __forceinline__ void rd_write_obs(const StepParams& P, const OutPtrs& o, const DevMap& m, int e, int map_id,
                                             const double (&q)[7], uint32_t episode, uint32_t agent_step, int was_reset,
                                             bool have_cs, double c, double s) {
  ObsVals ov;
  rd_obs_compute(P, m, e, map_id, q, episode, agent_step, was_reset, have_cs, c, s, ov);
  rd_obs_store(P, o, e, ov);
}

__device__ __forceinline__ void rd_write_scalars(const OutPtrs& o, int e, float reward, int done, double p, int lap,
                                                 double time, int flags) {
  if (o.reward) o.reward[e] = reward;
  if (o.done) o.done[e] = (uint8_t)done;
  if (o.progress) o.progress[e] = (float)p;
  if (o.lap) o.lap[e] = lap;
  if (o.time) o.time[e] = (float)time;
  if (o.flags) o.flags[e] = (uint8_t)flags;
  if (o.wrong_way) o.wrong_way[e] = (flags & RD_F_WRONG_WAY) ? 1 : 0;
  if (o.wall_collision) o.wall_collision[e] = (flags & RD_F_COLLISION) ? 1 : 0;
}

// K5 episode statistics: warp reduce, one atomic per warp and counter
// [REF dreamer/tools.py:159-206 simulate(): per-episode return / progress lists]
__device__ __forceinline__ void rd_stats_reduce(double* stats, const double (&st)[RD_NSTAT]) {
  const unsigned any_done = __ballot_sync(0xffffffffu, st[0] != 0.0);
#pragma unroll
  for (int k = 0; k < RD_NSTAT; ++k) {
    if (k != 6 && !any_done) continue;
    double v = st[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(stats + k, v);
  }
}

// keep_others: envs outside the mask are marked frozen (was_reset = 2: the LiDAR / occupancy kernels leave their rows as
// they are) instead of being observed again (3); their rows are the same either way (pose and noise counters unchanged)
__global__ void __launch_bounds__(128) k_reset(StepParams P, OutPtrs o, const uint8_t* __restrict__ mask, int mode,
                                               int keep_others) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // k_lidar may start its set-up (see launch_lidar_t)
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.n) return;
  bool sel = (!mask || mask[e]);
  if (mask && P.cfg.agents_per_world > 1) {  // a world resets as a whole [REF dreamer/tools.py:178-179]
    const int A = P.cfg.agents_per_world, b = e - e % A;
    for (int j = 0; j < A; ++j) sel = sel || mask[b + j];
  }
  const int2 jv = P.S.i2[e];
  const DevMap& m = P.maps[jv.y];
  double q[7], p = 0.0;
  uint32_t episode = (uint32_t)jv.x, agent_step = 0u;
  if (sel) {
    rd_reset_one(P, m, e, mode, episode, jv.y, q, p);
    episode += 1u;
  } else {
    const double2 xy = rd_ldp(P.S, RD_P_XY, e), sv = rd_ldp(P.S, RD_P_SV, e), yw = rd_ldp(P.S, RD_P_YW, e);
    q[0] = xy.x; q[1] = xy.y; q[2] = sv.x; q[3] = sv.y; q[4] = yw.x; q[5] = yw.y; q[6] = rd_ldp(P.S, RD_P_ST, e).x;
    agent_step = (uint32_t)P.S.i4[e].w;
  }
  rd_write_obs(P, o, m, e, jv.y, q, episode, agent_step, sel ? 1 : (keep_others ? 2 : 3), false, 0.0,
               0.0);  // 3: not reset here -> occupancy untouched
  if (sel) {
    rd_write_scalars(o, e, 0.f, 0, p, 1, 0.0, 0);
    if (o.rank) o.rank[e] = 1 + (P.cfg.agents_per_world > 1 ? e % P.cfg.agents_per_world : 0);  // refined by the first step
    if (o.opponents) o.opponents[e] = 0;
  }
}

// envs [e0, e1) of the batch (the host-facing path may step sub-ranges)
__global__ void __launch_bounds__(128) k_step(StepParams P, OutPtrs o, const float* __restrict__ actions, int e0, int e1) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // k_lidar may start its set-up (see launch_lidar_t)
  const int e = e0 + blockIdx.x * blockDim.x + threadIdx.x;
  const rd_config& cfg = P.cfg;
  const StateRef& S = P.S;
  double st[RD_NSTAT] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // rd_stats contributions of this env
  if (e < e1) {
    // Every load of this env's state is issued up front, before the first branch, as 128-bit requests: after a cold L2
    // (another kernel ran in between) each dependent round trip to HBM costs ~1 us of this latency-bound kernel.
    const int4 iv = S.i4[e];
    const int2 jv = S.i2[e];
    const float2 act = reinterpret_cast<const float2*>(actions)[e];
    const double2 pxy = rd_ldp(S, RD_P_XY, e), psv = rd_ldp(S, RD_P_SV, e), pyw = rd_ldp(S, RD_P_YW, e);
    const double2 pst = rd_ldp(S, RD_P_ST, e), ppl = rd_ldp(S, RD_P_PL, e), prs = rd_ldp(S, RD_P_RS, e);
    const double2 pmp = rd_ldp(S, RD_P_MP, e);
    int lap = iv.x, cp = iv.y, flags = iv.z;
    const int agent_step0 = iv.w, map_id = jv.y;
    double time = pst.y, p = ppl.x, last = ppl.y;
    if (flags & RD_F_NEEDS_RESET) {  // frozen until reset [REF dreamer/wrappers.py:148]
      rd_write_scalars(o, e, 0.f, 1, p, lap, time, flags);
      P.recs[e].was_reset = 2;
    } else {
      const DevMap m = P.maps[map_id];   // the track descriptor lives in registers for the whole step
      const double a0 = rd_action(cfg, act.x, 0), a1 = rd_action(cfg, act.y, 1);
      double q[7] = {pxy.x, pxy.y, psv.x, psv.y, pyw.x, pyw.y, pst.x};
      double total = 0.0;
      int done = 0, tick_timeout = 0;
      const int R = cfg.action_repeat;
      // ActionRepeat [REF dreamer/wrappers.py:107-116], software-pipelined: iteration t integrates tick t into qn while
      // the map loads of tick t-1's footprint probe are in flight, then does tick t-1's bookkeeping (lap machine, reward,
      // termination).  A tick integrated past a terminal one is discarded (q is only advanced after the test).
      Probe pr;
      double qn[7];
      double hc = 0.0, hs = 0.0;
#pragma unroll 1
      for (int t = 0; t <= R; ++t) {
        if (t < R) {
#pragma unroll
          for (int k = 0; k < 7; ++k) qn[k] = q[k];
          rdv_tick(P.vk, P.off, P.vk_g, P.off_g, qn, a0, a1);
        }
        if (t > 0) {
          time = time + cfg.dt;
          bool col, inside;
          rd_probe_finish(m, pr, col, inside, p);
          hc = pr.c; hs = pr.s;
          flags &= ~(RD_F_COLLISION | RD_F_LEFT_MAP);
          if (col) flags |= RD_F_COLLISION;
          if (!inside) flags |= RD_F_LEFT_MAP;
          if (!(q[0] == q[0] && q[1] == q[1] && q[3] == q[3] && q[4] == q[4])) flags |= RD_F_NAN;
          rd_lap_machine(cfg, p, lap, cp, flags);
          const double cur = (double)lap + p;
          bool d;
          const double r = rd_task_reward(cfg, cfg.task, col, cur, last, a1, q[3], q[6], lap, time, d);
          if (cfg.time_limit_ticks > 0 && agent_step0 * R + t >= cfg.time_limit_ticks) { tick_timeout = !d; d = true; }
          last = cur;
          total = total + r;
          // dreamer: stop at the first done [REF dreamer/wrappers.py:112]; baselines: the done of the first tick is not
          // tested when more ticks follow [REF baselines/racing/environment/single_agent.py:32-38]
          if (d && !(cfg.repeat_semantics == RD_REPEAT_BASELINES && t == 1 && R > 1)) { done = 1; break; }
          tick_timeout = 0;
        }
        if (t < R) {
#pragma unroll
          for (int k = 0; k < 7; ++k) q[k] = qn[k];
          rd_probe_issue(cfg, m, q[0], q[1], q[4], pr);
        }
      }
      const int agent_step = agent_step0 + 1;  // TimeLimit [REF dreamer/wrappers.py:147-154]
      int timeout = done ? tick_timeout : 0;
      if (cfg.time_limit_steps > 0 && agent_step >= cfg.time_limit_steps) { timeout = timeout || !done; done = 1; }
      const double ret = prs.x + total;
      const double epi = ((double)lap + p) - 1.0;           // tools.simulate's per-step progress [REF dreamer/tools.py:195]
      const double mp = epi > pmp.x ? epi : pmp.x;
      if (done && !cfg.auto_reset) flags |= RD_F_NEEDS_RESET;
      rd_write_scalars(o, e, (float)total, done, p, lap, time, flags);
      st[6] = 1.0;
      if (done) {
        st[0] = 1.0; st[1] = ret; st[2] = ((double)lap + p) - prs.y;
        st[3] = (double)agent_step; st[4] = (flags & RD_F_COLLISION) ? 1.0 : 0.0; st[5] = (double)(lap - 1);
        st[7] = timeout ? 1.0 : 0.0; st[8] = mp;
      }
      if (done && cfg.auto_reset) {
        double pz;
        rd_reset_one(P, m, e, cfg.reset_mode, (uint32_t)jv.x, map_id, q, pz);
        rd_write_obs(P, o, m, e, map_id, q, (uint32_t)jv.x + 1u, 0u, 1, false, 0.0, 0.0);
      } else {
        rd_stp(S, RD_P_XY, e, q[0], q[1]);
        rd_stp(S, RD_P_SV, e, q[2], q[3]);
        rd_stp(S, RD_P_YW, e, q[4], q[5]);
        rd_stp(S, RD_P_ST, e, q[6], time);
        rd_stp(S, RD_P_PL, e, p, last);
        rd_stp(S, RD_P_RS, e, ret, prs.y);
        rd_stp(S, RD_P_MP, e, mp, 0.0);
        S.i4[e] = make_int4(lap, cp, flags, agent_step);
        rd_write_obs(P, o, m, e, map_id, q, (uint32_t)jv.x, (uint32_t)agent_step, 0, true, hc, hs);
      }
    }
  }
  rd_stats_reduce(P.stats, st);
}

// k_step over FOUR warps per 32 envs.  k_step's time is the latency of one env's in-order instruction stream (one warp
// per SM sub-partition), and that stream holds chains that only feed FORWARD:
//   warp 0 "dynamics"     the five coupled vehicle states, four dependent RK4 stages per tick, for all R ticks;
//   warp 1 "position"     four sine/cosine pairs per tick on the stage headings those leave behind -> x, y;
//   warp 2 "probe"        cosine/sine of the new heading, the footprint's five cells, their bit-grid / wavefront loads
//                         (issued for tick t, stored while tick t+1's arithmetic runs); after the last tick it writes the
//                         observation scalars and the LiDAR origin record of the state after R ticks -- what the step
//                         returns unless the env finishes, which warp 3 then overwrites;
//   warp 3 "bookkeeping"  k_step's own per-tick body (lap machine, reward, termination) on what the rings hold, then
//                         scalars, commit, statistics, and the observation of the envs that finished or were reset;
//   warp 4 "reset"        (auto-reset only) looks up, right at the start, the pose every env WOULD be reset to -- a
//                         pure function of (env, episode) -- with its progress and its observation record: three
//                         dependent map loads and a general sine/cosine that would otherwise sit, for the few lanes
//                         that finish, at the very end of their whole warp's critical path (88 of 128 CTAs had such a
//                         lane in a config-2 step; it cost them 3.6 us).
// One mbarrier per tick and ring, no back-pressure (the rings hold all R <= RD_SPLIT_TICKS ticks).  Same arithmetic,
// operation for operation, as k_step (rdv_tick_core_t + rdv_tick_position are what rdv_tick_t is made of); ticks
// integrated past a terminal one are simply never read.
#define RD_SPLIT_TICKS 8
#define RD_SPLIT_FIELDS 13   // ring 0: ang[4], vs[4], steer, v, yaw, yaw_rate, slip
#define RD_SPLIT_PROBE 8     // ring 2: five bit-grid words, the centre's wavefront distance, shifts + inside flag
__device__ __forceinline__ void rd_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(rd_smem_u32(bar)) : "memory");   // release.cta
}
#ifdef RD_SPLIT_TRACE   // tuning: per-warp time stamps (cycles since the CTA started) of one CTA, printed at the end
#define RD_TR(i) do { if (lane == 0 && blockIdx.x == 5 && (i) < 24) tr[warp][(i)] = clock64() - t_begin; } while (0)
#define RD_TR_DUMP(n) do { if (lane == 0 && blockIdx.x == 5) { printf("[k_step_split warp %d]", warp); for (int i_ = 0; i_ < (n); ++i_) printf(" %lld", tr[warp][i_]); printf("\n"); } } while (0)
#else
#define RD_TR(i) do {} while (0)
#define RD_TR_DUMP(n) do {} while (0)
#endif
__global__ void __launch_bounds__(160) k_step_split(StepParams P, OutPtrs o, const float* __restrict__ actions, int e0, int e1) {
#ifdef RD_SPLIT_TRACE
  __shared__ long long tr[4][24];
  const long long t_begin = clock64();
#endif
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // k_lidar may start its set-up (see launch_lidar_t)
  __shared__ __align__(16) double rg[RD_SPLIT_TICKS][RD_SPLIT_FIELDS][32];   // 26 KB  warp 0 -> 1, 2, 3
  __shared__ __align__(16) double rp[RD_SPLIT_TICKS][2][32];                 // 4 KB   warp 1 -> 2, 3: x, y
  __shared__ __align__(16) double rc[RD_SPLIT_TICKS][2][32];                 // 4 KB   warp 2 -> 3: cos, sin of the heading
  __shared__ __align__(16) uint32_t rq[RD_SPLIT_TICKS][RD_SPLIT_PROBE][32];  // 8 KB   warp 2 -> 3: the probe
  __shared__ __align__(16) double rs[4][32];                                 // 1 KB   warp 4 -> 3: reset pose x, y, yaw, progress
  __shared__ __align__(16) uint32_t ro[RD_OBS_WORDS][32];                    // 3 KB   warp 4 -> 3: its observation (ObsVals)
  __shared__ __align__(8) uint64_t fb[3][RD_SPLIT_TICKS];
  __shared__ __align__(8) uint64_t obs_bar, rst_bar;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = e0 + blockIdx.x * 32 + lane;
  const rd_config& cfg = P.cfg;
  const StateRef& S = P.S;
  const int R = cfg.action_repeat;
  if (threadIdx.x < 3 * RD_SPLIT_TICKS) rd_mbar_init(&fb[0][0] + threadIdx.x, 32);
  if (threadIdx.x == 3 * RD_SPLIT_TICKS) { rd_mbar_init(&obs_bar, 32); rd_mbar_init(&rst_bar, 32); }
  __syncthreads();
  if (warp == 4) {
    // ---- reset warp ----
    if (cfg.auto_reset && e < e1) {
      const int2 jv = S.i2[e];
      const DevMap m = P.maps[jv.y];
      double x, y, yaw, p;
      rd_reset_pose(P, m, e, cfg.reset_mode, (uint32_t)jv.x, x, y, yaw, p);
      const double q[7] = {x, y, 0.0, 0.0, yaw, 0.0, 0.0};
      ObsVals ov;
      rd_obs_compute(P, m, e, jv.y, q, (uint32_t)jv.x + 1u, 0u, 1, false, 0.0, 0.0, ov);
      rs[0][lane] = x; rs[1][lane] = y; rs[2][lane] = yaw; rs[3][lane] = p;
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&ov);
#pragma unroll
      for (int k = 0; k < RD_OBS_WORDS; ++k) ro[k][lane] = w[k];
    }
    rd_mbar_arrive(&rst_bar);
    return;
  }
  if (warp == 0) {
    // ---- dynamics warp ----
    bool live = false;
    double q[7] = {0, 0, 0, 0, 0, 0, 0};
    double a0 = 0.0, a1 = 0.0;
    if (e < e1) {
      const int4 iv = S.i4[e];
      const float2 act = reinterpret_cast<const float2*>(actions)[e];
      const double2 psv = rd_ldp(S, RD_P_SV, e), pyw = rd_ldp(S, RD_P_YW, e), pst = rd_ldp(S, RD_P_ST, e);
      live = !(iv.z & RD_F_NEEDS_RESET);
      a0 = rd_action(cfg, act.x, 0); a1 = rd_action(cfg, act.y, 1);
      q[2] = psv.x; q[3] = psv.y; q[4] = pyw.x; q[5] = pyw.y; q[6] = pst.x;
    }
    RD_TR(0);
#pragma unroll 1
    for (int t = 0; t < R; ++t) {
      if (live) {
        double ang[4], vs[4];
        rdv_tick_core(P.vk, P.off, P.vk_g, P.off_g, q, a0, a1, ang, vs);
#pragma unroll
        for (int k = 0; k < 4; ++k) { rg[t][k][lane] = ang[k]; rg[t][4 + k][lane] = vs[k]; }
#pragma unroll
        for (int k = 0; k < 5; ++k) rg[t][8 + k][lane] = q[2 + k];
      }
      rd_mbar_arrive(&fb[0][t]);
      RD_TR(1 + t);
    }
    RD_TR_DUMP(1 + R);
    return;
  }
  if (warp == 1) {
    // ---- position warp ----
    bool live = false;
    double x = 0.0, y = 0.0;
    if (e < e1) {
      const int4 iv = S.i4[e];
      const double2 pxy = rd_ldp(S, RD_P_XY, e);
      live = !(iv.z & RD_F_NEEDS_RESET);
      x = pxy.x; y = pxy.y;
    }
#pragma unroll 1
    for (int t = 0; t < R; ++t) {
      rd_mbar_wait(&fb[0][t], 0);
      if (live) {
        double ang[4], vs[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { ang[k] = rg[t][k][lane]; vs[k] = rg[t][4 + k][lane]; }
        // the short trigonometric path when every argument is in its range (always, unless a car has spun thousands of
        // times): four independent chains in one straight-line block
        const bool in_range = fabs(ang[0]) < 1.0e5 && fabs(ang[1]) < 1.0e5 && fabs(ang[2]) < 1.0e5 && fabs(ang[3]) < 1.0e5;
        if (in_range) rdv_tick_position<true>(P.vk, ang, vs, x, y);
        else rdv_tick_position<false>(P.vk, ang, vs, x, y);
        rp[t][0][lane] = x; rp[t][1][lane] = y;
      }
      rd_mbar_arrive(&fb[1][t]);
      RD_TR(1 + t);
    }
    RD_TR_DUMP(1 + R);
    return;
  }
  if (warp == 2) {
    // ---- probe warp ----
    bool live = false;
    int map_id = 0, episode = 0, agent_step0 = 0;
    if (e < e1) {
      const int4 iv = S.i4[e];
      const int2 jv = S.i2[e];
      live = !(iv.z & RD_F_NEEDS_RESET);
      agent_step0 = iv.w; episode = jv.x; map_id = jv.y;
    }
    const DevMap m = P.maps[map_id];
    Probe pr{};
    double qf[7] = {0, 0, 0, 0, 0, 0, 0};
    auto publish = [&](int t) {
      if (live) {
        rc[t][0][lane] = pr.c; rc[t][1][lane] = pr.s;
#pragma unroll
        for (int k = 0; k < 5; ++k) rq[t][k][lane] = pr.w[k];
        rq[t][5][lane] = pr.dval;
        rq[t][6][lane] = (uint32_t)pr.sh[0] | ((uint32_t)pr.sh[1] << 5) | ((uint32_t)pr.sh[2] << 10) | ((uint32_t)pr.sh[3] << 15) |
                         ((uint32_t)pr.sh[4] << 20) | (pr.in0 ? 0x80000000u : 0u);
      }
      rd_mbar_arrive(&fb[2][t]);
    };
#pragma unroll 1
    for (int t = 0; t < R; ++t) {
      rd_mbar_wait(&fb[0][t], 0);
      RD_TR(1 + t);
      double c = 1.0, s = 0.0;
      if (live) rdv_sincos(rg[t][10][lane], s, c);   // the new heading: in flight while the position warp finishes tick t
      rd_mbar_wait(&fb[1][t], 0);
      if (t > 0) publish(t - 1);                     // tick t-1's loads have had this tick's trigonometry to arrive
      if (live) {
        qf[0] = rp[t][0][lane]; qf[1] = rp[t][1][lane];
        rd_probe_issue_cs(cfg, m, qf[0], qf[1], c, s, pr);
      }
    }
    publish(R - 1);
    RD_TR(10);
    if (live) {   // the observation of the state after R ticks (warp 3 overwrites it for the envs that finish)
#pragma unroll
      for (int k = 0; k < 5; ++k) qf[2 + k] = rg[R - 1][8 + k][lane];
      rd_write_obs(P, o, m, e, map_id, qf, (uint32_t)episode, (uint32_t)(agent_step0 + 1), 0, true, pr.c, pr.s);
    }
    rd_mbar_arrive(&obs_bar);
    RD_TR(11);
    RD_TR_DUMP(12);
    return;
  }
  // ---- bookkeeping warp: k_step with the tick integration replaced by the ring ----
  double st[RD_NSTAT] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // rd_stats contributions of this env
  if (e < e1) {
    const int4 iv = S.i4[e];
    const int2 jv = S.i2[e];
    const float2 act = reinterpret_cast<const float2*>(actions)[e];
    const double2 pxy = rd_ldp(S, RD_P_XY, e), psv = rd_ldp(S, RD_P_SV, e), pyw = rd_ldp(S, RD_P_YW, e);
    const double2 pst = rd_ldp(S, RD_P_ST, e), ppl = rd_ldp(S, RD_P_PL, e), prs = rd_ldp(S, RD_P_RS, e);
    const double2 pmp = rd_ldp(S, RD_P_MP, e);
    int lap = iv.x, cp = iv.y, flags = iv.z;
    const int agent_step0 = iv.w, map_id = jv.y;
    double time = pst.y, p = ppl.x, last = ppl.y;
    if (flags & RD_F_NEEDS_RESET) {  // frozen until reset [REF dreamer/wrappers.py:148]
      rd_write_scalars(o, e, 0.f, 1, p, lap, time, flags);
      P.recs[e].was_reset = 2;
    } else {
      const DevMap m = P.maps[map_id];   // the track descriptor lives in registers for the whole step
      RD_TR(0);
      const double a1 = rd_action(cfg, act.y, 1);
      double q[7] = {pxy.x, pxy.y, psv.x, psv.y, pyw.x, pyw.y, pst.x};
      double total = 0.0;
      int done = 0, tick_timeout = 0;
      double hc = 0.0, hs = 0.0;
#pragma unroll 1
      for (int t = 1; t <= R; ++t) {      // t ticks done, as in k_step's bookkeeping half
        rd_mbar_wait(&fb[2][t - 1], 0);   // acquire: the probe warp's tick (and with it the other two warps') is there
        Probe pr;
        q[0] = rp[t - 1][0][lane]; q[1] = rp[t - 1][1][lane]; pr.c = rc[t - 1][0][lane]; pr.s = rc[t - 1][1][lane];
#pragma unroll
        for (int k = 0; k < 5; ++k) q[2 + k] = rg[t - 1][8 + k][lane];
#pragma unroll
        for (int k = 0; k < 5; ++k) pr.w[k] = rq[t - 1][k][lane];
        pr.dval = rq[t - 1][5][lane];
        const uint32_t packed = rq[t - 1][6][lane];
#pragma unroll
        for (int k = 0; k < 5; ++k) pr.sh[k] = (int)((packed >> (5 * k)) & 31u);
        pr.in0 = (packed >> 31) != 0u;
        time = time + cfg.dt;
        bool col, inside;
        rd_probe_finish(m, pr, col, inside, p);
        hc = pr.c; hs = pr.s;
        flags &= ~(RD_F_COLLISION | RD_F_LEFT_MAP);
        if (col) flags |= RD_F_COLLISION;
        if (!inside) flags |= RD_F_LEFT_MAP;
        if (!(q[0] == q[0] && q[1] == q[1] && q[3] == q[3] && q[4] == q[4])) flags |= RD_F_NAN;
        rd_lap_machine(cfg, p, lap, cp, flags);
        const double cur = (double)lap + p;
        bool d;
        const double r = rd_task_reward(cfg, cfg.task, col, cur, last, a1, q[3], q[6], lap, time, d);
        if (cfg.time_limit_ticks > 0 && agent_step0 * R + t >= cfg.time_limit_ticks) { tick_timeout = !d; d = true; }
        last = cur;
        total = total + r;
        // dreamer: stop at the first done [REF dreamer/wrappers.py:112]; baselines: the done of the first tick is not
        // tested when more ticks follow [REF baselines/racing/environment/single_agent.py:32-38]
        if (d && !(cfg.repeat_semantics == RD_REPEAT_BASELINES && t == 1 && R > 1)) { done = 1; break; }
        tick_timeout = 0;
        RD_TR(1 + t);
      }
      const int agent_step = agent_step0 + 1;  // TimeLimit [REF dreamer/wrappers.py:147-154]
      int timeout = done ? tick_timeout : 0;
      if (cfg.time_limit_steps > 0 && agent_step >= cfg.time_limit_steps) { timeout = timeout || !done; done = 1; }
      const double ret = prs.x + total;
      const double epi = ((double)lap + p) - 1.0;           // tools.simulate's per-step progress [REF dreamer/tools.py:195]
      const double mp = epi > pmp.x ? epi : pmp.x;
      if (done && !cfg.auto_reset) flags |= RD_F_NEEDS_RESET;
      rd_write_scalars(o, e, (float)total, done, p, lap, time, flags);
      st[6] = 1.0;
      if (done) {
        st[0] = 1.0; st[1] = ret; st[2] = ((double)lap + p) - prs.y;
        st[3] = (double)agent_step; st[4] = (flags & RD_F_COLLISION) ? 1.0 : 0.0; st[5] = (double)(lap - 1);
        st[7] = timeout ? 1.0 : 0.0; st[8] = mp;
      }
      if (done) rd_mbar_wait(&obs_bar, 0);   // the probe warp's observation of the R-tick state is out: what follows replaces it
      if (done && cfg.auto_reset) {
        rd_mbar_wait(&rst_bar, 0);           // the reset warp's pose and observation for this (env, episode)
        rd_reset_commit(P, e, (uint32_t)jv.x, map_id, rs[0][lane], rs[1][lane], rs[2][lane], rs[3][lane], q);
        ObsVals ov;
        uint32_t* w = reinterpret_cast<uint32_t*>(&ov);
#pragma unroll
        for (int k = 0; k < RD_OBS_WORDS; ++k) w[k] = ro[k][lane];
        rd_obs_store(P, o, e, ov);
      } else {
        rd_stp(S, RD_P_XY, e, q[0], q[1]);
        rd_stp(S, RD_P_SV, e, q[2], q[3]);
        rd_stp(S, RD_P_YW, e, q[4], q[5]);
        rd_stp(S, RD_P_ST, e, q[6], time);
        rd_stp(S, RD_P_PL, e, p, last);
        rd_stp(S, RD_P_RS, e, ret, prs.y);
        rd_stp(S, RD_P_MP, e, mp, 0.0);
        S.i4[e] = make_int4(lap, cp, flags, agent_step);
        // not done: all R ticks ran and the probe warp has written exactly this observation already
        if (done) rd_write_obs(P, o, m, e, map_id, q, (uint32_t)jv.x, (uint32_t)agent_step, 0, true, hc, hs);
      }
    }
  }
  RD_TR(12);
  RD_TR_DUMP(13);
#ifdef RD_SPLIT_TRACE
  { const unsigned dn = __ballot_sync(0xffffffffu, st[0] != 0.0); if (lane == 0) printf("[cta %d] end %lld done %08x\n", blockIdx.x, clock64() - t_begin, dn); }
#endif
  rd_stats_reduce(P.stats, st);
}

// ---- multi-agent worlds (SURVEY.md §8-f3) -----------------------------------------------------------------------
// Overlap of two body boxes (half extents hl x hw, centres d apart, headings (c1,s1), (c2,s2)): separating-axis test on
// the four box axes, float64, one IEEE operation per step in the order written (the oracle's rect_overlap).
// [NEW-SPEC: racecar_gym reports Bullet contacts between racecars as info['opponent_collisions']]
__device__ __forceinline__ bool rd_rect_overlap(double hl, double hw, double dx, double dy, double c1, double s1,
                                                double c2, double s2) {
  const double cr = fabs(c1 * c2 + s1 * s2), sr = fabs(c1 * s2 - s1 * c2);
  const double ex = hl + (hl * cr + hw * sr), ey = hw + (hl * sr + hw * cr);
  if (fabs(dx * c1 + dy * s1) > ex) return false;
  if (fabs(dy * c1 - dx * s1) > ey) return false;
  if (fabs(dx * c2 + dy * s2) > ex) return false;
  if (fabs(dy * c2 - dx * s2) > ey) return false;
  return true;
}

// k_step for worlds of A = cfg.agents_per_world cars (A = 1 allowed: single cars on the n_step_progress task).
// One thread per car; the cars of a world are adjacent threads of one CTA (a CTA holds blockDim.x / A whole worlds) and
// exchange poses / done flags through shared memory every tick:
//   tick:  every car integrates its own dynamics and probes the walls            -> pose to shared memory
//          body-box overlap with the other cars of the world (opponent mask), progress/lap machine, the car's own task
//          reward and done                                                        -> done flag to shared memory
//          dreamer ActionRepeat: the WORLD stops repeating at the first tick in which any car is done
//          [REF dreamer/wrappers.py:112]; baselines multi-agent ActionRepeat: all ticks run, dones are OR-ed
//          [REF baselines/racing/environment/multi_agent.py:72-79]; a single car under the baselines semantics follows
//          single_agent.py's rule like k_step (the first tick's done is not tested, a later one stops the repeat)
//   then:  TimeLimit (one counter per world, all dones True [REF dreamer/wrappers.py:151-153]), rank, commit, auto-reset
//          of the whole world when any car is done [REF dreamer/tools.py:178-179].
// Episode statistics follow tools.simulate: the world's first agent only [REF dreamer/tools.py:162-165 main_id].
__global__ void __launch_bounds__(128) k_step_ma(StepParams P, OutPtrs o, const float* __restrict__ actions) {
  __shared__ double sh_pose[128 * 4];
  __shared__ double sh_prog[128];
  __shared__ int sh_flag[128];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // k_lidar may start its set-up (see launch_lidar_t)
  const int n = P.n;
  const rd_config& cfg = P.cfg;
  const StateRef& S = P.S;
  const int A = cfg.agents_per_world > 1 ? cfg.agents_per_world : 1;
  const int wpc = (int)blockDim.x / A;             // worlds per CTA
  const int t = (int)threadIdx.x;
  const int e = (int)blockIdx.x * wpc * A + t;
  const bool live = t < wpc * A && e < n;
  const int a = t % A, base = t - a;               // agent index, first thread of my world
  double st[RD_NSTAT] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int4 iv = make_int4(1, 0, 0, 0);
  int2 jv = make_int2(0, 0);
  if (live) { iv = S.i4[e]; jv = S.i2[e]; }
  int flags = iv.z;
  const bool frozen = live && (flags & RD_F_NEEDS_RESET);
  const bool run = live && !frozen;
  const int task = A > 1 ? cfg.agent_task[a] : cfg.task;
  const bool ma_or = cfg.repeat_semantics == RD_REPEAT_BASELINES && A > 1;    // multi_agent.py: run every tick, OR the dones
  const bool sa_skip = cfg.repeat_semantics == RD_REPEAT_BASELINES && A == 1; // single_agent.py: the first tick's done is not tested
  const int R = cfg.action_repeat;
  const double hl = 0.5 * cfg.vehicle.body_length, hw = 0.5 * cfg.vehicle.body_width;
  const int map_id = run ? jv.y : 0;
  const DevMap m = P.maps[map_id];
  double act[2] = {0.0, 0.0};
  double q[7] = {0, 0, 0, 0, 0, 0, 0};
  double time = 0.0, p = 0.0, last = 0.0, total = 0.0, ret0 = 0.0, start0 = 0.0, mp0 = 0.0, hc = 1.0, hs = 0.0;
  int lap = iv.x, cp = iv.y, opp = 0, done = 0, tick_timeout = 0;
  const int agent_step0 = iv.w;
  if (run) {
    const float2 af = reinterpret_cast<const float2*>(actions)[e];
    act[0] = rd_action(cfg, af.x, 0); act[1] = rd_action(cfg, af.y, 1);
    const double2 pxy = rd_ldp(S, RD_P_XY, e), psv = rd_ldp(S, RD_P_SV, e), pyw = rd_ldp(S, RD_P_YW, e);
    const double2 pst = rd_ldp(S, RD_P_ST, e), ppl = rd_ldp(S, RD_P_PL, e), prs = rd_ldp(S, RD_P_RS, e);
    q[0] = pxy.x; q[1] = pxy.y; q[2] = psv.x; q[3] = psv.y; q[4] = pyw.x; q[5] = pyw.y; q[6] = pst.x;
    time = pst.y; p = ppl.x; last = ppl.y; ret0 = prs.x; start0 = prs.y; mp0 = rd_ldp(S, RD_P_MP, e).x;
  } else if (frozen) {
    const double2 pst = rd_ldp(S, RD_P_ST, e), ppl = rd_ldp(S, RD_P_PL, e);
    time = pst.y; p = ppl.x;
  }
  bool ticking = run;
  for (int tk = 0; tk < R; ++tk) {
    bool col = false, inside = true;
    if (ticking) {
      rdv_tick(P.vk, P.off, P.vk_g, P.off_g, q, act[0], act[1]);
      time = time + cfg.dt;
      Probe pr;
      rd_probe_issue(cfg, m, q[0], q[1], q[4], pr);
      rd_probe_finish(m, pr, col, inside, p);
      hc = pr.c; hs = pr.s;
      sh_pose[4 * t] = q[0]; sh_pose[4 * t + 1] = q[1]; sh_pose[4 * t + 2] = hc; sh_pose[4 * t + 3] = hs;
    }
    __syncthreads();
    int d = 0;
    if (ticking) {
      opp = 0;
      for (int j = 0; j < A; ++j) {
        if (j == a) continue;
        const double* w = sh_pose + 4 * (base + j);
        if (rd_rect_overlap(hl, hw, w[0] - q[0], w[1] - q[1], hc, hs, w[2], w[3])) opp |= 1 << j;
      }
      flags &= ~(RD_F_COLLISION | RD_F_LEFT_MAP | RD_F_OPPONENT);
      if (col) flags |= RD_F_COLLISION;
      if (opp) flags |= RD_F_OPPONENT;
      if (!inside) flags |= RD_F_LEFT_MAP;
      if (!(q[0] == q[0] && q[1] == q[1] && q[3] == q[3] && q[4] == q[4])) flags |= RD_F_NAN;
      const bool hitc = col || opp != 0;   // the task's collision: walls or other cars
      rd_lap_machine(cfg, p, lap, cp, flags);
      const double cur = (double)lap + p;
      double ref = last;
      if (task == RD_TASK_N_STEP_PROGRESS && P.hist) {  // progress over the last n ticks
        const int slot = (agent_step0 * R + tk) % cfg.n_step_progress;
        ref = P.hist[(size_t)slot * n + e];
        P.hist[(size_t)slot * n + e] = cur;
      }
      bool db;
      const double r = rd_task_reward(cfg, task, hitc, cur, ref, act[1], q[3], q[6], lap, time, db);
      int tto = 0;
      if (cfg.time_limit_ticks > 0 && agent_step0 * R + tk + 1 >= cfg.time_limit_ticks) { tto = !db; db = true; }
      last = cur;
      total = total + r;
      if (ma_or) { d = db ? 1 : 0; done |= d; tick_timeout |= tto; d = 0; }
      else { d = (db && !(sa_skip && tk == 0 && R > 1)) ? 1 : 0; done = d; tick_timeout = d ? tto : 0; }
      sh_flag[t] = d;
    }
    __syncthreads();
    if (ticking) {
      int any = 0;
      for (int j = 0; j < A; ++j) any |= sh_flag[base + j];
      if (any) ticking = false;
    }
  }
  // world-level done, rank
  __syncthreads();
  if (run) { sh_flag[t] = done; sh_prog[t] = (double)lap + p; }
  __syncthreads();
  if (frozen) {  // frozen until reset [REF dreamer/wrappers.py:148]
    rd_write_scalars(o, e, 0.f, 1, p, lap, time, flags);
    P.recs[e].was_reset = 2;
  } else if (run) {
    int wdone = 0, rank = 1;
    const double mine = sh_prog[t];
    for (int j = 0; j < A; ++j) {
      wdone |= sh_flag[base + j];
      if (j != a) { const double other = sh_prog[base + j]; if (other > mine || (other == mine && j < a)) rank += 1; }
    }
    const int agent_step = agent_step0 + 1;  // TimeLimit [REF dreamer/wrappers.py:147-154]
    int timeout = done ? tick_timeout : 0;
    if (cfg.time_limit_steps > 0 && agent_step >= cfg.time_limit_steps) { timeout = timeout || !wdone; done = 1; wdone = 1; }
    const double ret = ret0 + total;
    const double epi = ((double)lap + p) - 1.0;
    const double mp = epi > mp0 ? epi : mp0;
    if (wdone && !cfg.auto_reset) flags |= RD_F_NEEDS_RESET;
    rd_write_scalars(o, e, (float)total, done, p, lap, time, flags);
    if (o.rank) o.rank[e] = rank;
    if (o.opponents) o.opponents[e] = (uint8_t)opp;
    st[6] = 1.0;
    if (wdone && a == 0) {
      st[0] = 1.0; st[1] = ret; st[2] = ((double)lap + p) - start0;
      st[3] = (double)agent_step; st[4] = (flags & (RD_F_COLLISION | RD_F_OPPONENT)) ? 1.0 : 0.0; st[5] = (double)(lap - 1);
      st[7] = timeout ? 1.0 : 0.0; st[8] = mp;
    }
    if (wdone && cfg.auto_reset) {
      double pz;
      rd_reset_one(P, m, e, cfg.reset_mode, (uint32_t)jv.x, map_id, q, pz);
      rd_write_obs(P, o, m, e, map_id, q, (uint32_t)jv.x + 1u, 0u, 1, false, 0.0, 0.0);
    } else {
      rd_stp(S, RD_P_XY, e, q[0], q[1]);
      rd_stp(S, RD_P_SV, e, q[2], q[3]);
      rd_stp(S, RD_P_YW, e, q[4], q[5]);
      rd_stp(S, RD_P_ST, e, q[6], time);
      rd_stp(S, RD_P_PL, e, p, last);
      rd_stp(S, RD_P_RS, e, ret, start0);
      rd_stp(S, RD_P_MP, e, mp, 0.0);
      S.i4[e] = make_int4(lap, cp, flags, agent_step);
      rd_write_obs(P, o, m, e, map_id, q, (uint32_t)jv.x, (uint32_t)agent_step, 0, true, hc, hs);
    }
  }
  rd_stats_reduce(P.stats, st);
}

// a1 stage entry: dynamics only, state [7][n] SoA, commands [n][2] sim-facing (rd_dynamics)
__global__ void __launch_bounds__(128) k_dynamics(VehConst vk, VehAcc off, const VehConst* __restrict__ vk_g,
                                                   const VehAcc* __restrict__ off_g, double* __restrict__ state,
                                                   const double* __restrict__ commands, int n, int n_ticks) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  double q[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) q[k] = state[(size_t)k * n + e];
  const double motor = commands[2 * e], steering = commands[2 * e + 1];
#pragma unroll 1
  for (int t = 0; t < n_ticks; ++t) rdv_tick(vk, off, vk_g, off_g, q, motor, steering);
#pragma unroll
  for (int k = 0; k < 7; ++k) state[(size_t)k * n + e] = q[k];
}

// a7/a8 stage entry (rd_reward_done): one tick of bookkeeping + task reward/done for teacher-forced poses
__global__ void __launch_bounds__(128) k_reward_done(rd_config cfg, const DevMap* __restrict__ maps,
                                                      const int32_t* __restrict__ map_ids, const double* __restrict__ kin,
                                                      const double* __restrict__ steering, int n,
                                                      double* __restrict__ book_f64, int32_t* __restrict__ book_i32,
                                                      double* __restrict__ reward, uint8_t* __restrict__ done) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const DevMap m = maps[map_ids ? map_ids[e] : 0];
  const double x = kin[e], y = kin[(size_t)n + e], yaw = kin[(size_t)2 * n + e], v = kin[(size_t)3 * n + e];
  const double slip = kin[(size_t)4 * n + e];
  double time = book_f64[e] + cfg.dt, p = book_f64[(size_t)n + e], last = book_f64[(size_t)2 * n + e];
  int lap = book_i32[e], cp = book_i32[(size_t)n + e], flags = book_i32[(size_t)2 * n + e];
  Probe pr;
  rd_probe_issue(cfg, m, x, y, yaw, pr);
  bool col, inside;
  rd_probe_finish(m, pr, col, inside, p);
  flags &= ~(RD_F_COLLISION | RD_F_LEFT_MAP);
  if (col) flags |= RD_F_COLLISION;
  if (!inside) flags |= RD_F_LEFT_MAP;
  if (!(x == x && y == y && v == v && yaw == yaw)) flags |= RD_F_NAN;
  rd_lap_machine(cfg, p, lap, cp, flags);
  const double cur = (double)lap + p;
  bool d;
  const double r = rd_task_reward(cfg, cfg.task, col, cur, last, steering ? steering[e] : 0.0, v, slip, lap, time, d);
  book_f64[e] = time; book_f64[(size_t)n + e] = p; book_f64[(size_t)2 * n + e] = cur;
  book_i32[e] = lap; book_i32[(size_t)n + e] = cp; book_i32[(size_t)2 * n + e] = flags;
  reward[e] = r;
  done[e] = d ? 1 : 0;
}

// rd_get_state / rd_set_state: the ABI's [RD_NF64][n] / [RD_NI32][n] layout <-> the internal 16-byte groups
__global__ void k_state_export(StateRef S, double* __restrict__ f64, int32_t* __restrict__ i32) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = S.n;
  if (e >= n) return;
  if (f64) {
#pragma unroll
    for (int k = 0; k < RD_NPAIR; ++k) {
      const double2 v = rd_ldp(S, k, e);
      f64[(size_t)(2 * k) * n + e] = v.x;
      if (2 * k + 1 < RD_NF64) f64[(size_t)(2 * k + 1) * n + e] = v.y;
    }
  }
  if (i32) {
    const int4 a = S.i4[e];
    const int2 b = S.i2[e];
    i32[(size_t)RD_I_LAP * n + e] = a.x; i32[(size_t)RD_I_CHECKPOINT * n + e] = a.y; i32[(size_t)RD_I_FLAGS * n + e] = a.z;
    i32[(size_t)RD_I_AGENT_STEP * n + e] = a.w; i32[(size_t)RD_I_EPISODE * n + e] = b.x; i32[(size_t)RD_I_MAP * n + e] = b.y;
  }
}
// the map column is owned by rd_assign_maps (the env grouping depends on it) and is not imported; restoring the float64
// part restarts the n_step_progress ring from the restored lap + progress
__global__ void k_state_import(StateRef S, const double* __restrict__ f64, const int32_t* __restrict__ i32,
                               double* __restrict__ hist, int n_hist) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = S.n;
  if (e >= n) return;
  if (f64) {
#pragma unroll
    for (int k = 0; k < RD_NPAIR; ++k)
      rd_stp(S, k, e, f64[(size_t)(2 * k) * n + e], (2 * k + 1 < RD_NF64) ? f64[(size_t)(2 * k + 1) * n + e] : 0.0);
    if (hist) for (int k = 0; k < n_hist; ++k) hist[(size_t)k * n + e] = f64[(size_t)RD_S_LAST * n + e];
  }
  if (i32) {
    S.i4[e] = make_int4(i32[(size_t)RD_I_LAP * n + e], i32[(size_t)RD_I_CHECKPOINT * n + e], i32[(size_t)RD_I_FLAGS * n + e],
                        i32[(size_t)RD_I_AGENT_STEP * n + e]);
    S.i2[e].x = i32[(size_t)RD_I_EPISODE * n + e];
  }
}
