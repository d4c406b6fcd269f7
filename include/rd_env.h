/* rd_env.h -- C ABI of the B200-native batched racing-environment step (librd_env.so).
 *
 * This is the drop-in boundary of SURVEY.md §8-b.  Every entry point names the reference interface it
 * replaces (paths relative to the reference tree, CPS-TUWien/racing_dreamer).  The arithmetic behind
 * a1/a2/a7/a8 lives in the un-vendored racecar_gym + PyBullet in the reference; the call sites cited here
 * are where the reference's Python reaches it.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++ or torch types cross this boundary.
 *   - every `*_dev` pointer is a CUDA device pointer owned by the CALLER (e.g. a torch tensor's data_ptr);
 *     `*_host` pointers are host memory.  The library owns only the handle, the env state and the maps.
 *   - all calls return 0 on success or a negative rd_status; rd_last_error() gives the sticky message.
 *   - calls taking `stream` (a cudaStream_t passed as void*) are asynchronous on that stream.
 *   - a handle is bound to the CUDA device current at rd_create and is not thread-safe.
 */
#ifndef RD_ENV_H
#define RD_ENV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RD_ABI_VERSION 3
#define RD_MAX_AGENTS 4   /* cars per world: agents A..D [REF baselines/scenarios/max_progress/austria.yml:3-34] */
#define RD_MAX_NSTEP 32   /* longest n of the n_step_progress task */

typedef struct rd_env rd_env; /* opaque */

typedef enum rd_status {
  RD_OK = 0,
  RD_ERR_INVALID = -1,   /* bad argument / configuration */
  RD_ERR_CUDA = -2,      /* CUDA runtime error (message has the cudaError string) */
  RD_ERR_STATE = -3,     /* call order: maps not uploaded / not assigned / not reset */
  RD_ERR_NOMEM = -4,
  RD_ERR_NO_DEVICE = -5  /* no usable sm_100 device: there is NO CPU fallback */
} rd_status;

/* reset modes [REF dreamer/wrappers.py:86-92 FixedResetMode; dreamer/dream.py:105-108,120] */
enum { RD_RESET_GRID = 0, RD_RESET_RANDOM = 1, RD_RESET_RANDOM_BIDIRECTIONAL = 2,
       RD_RESET_RANDOM_BALL = 3 /* multi-agent training: the cars of a world close to one random point
                                   [REF dreamer/dream.py:105-106] */ };
/* tasks [REF dreamer/scenarios/max_progress/austria.yml:8-10; baselines/racing/environment/tasks.py:4-22] */
enum { RD_TASK_MAX_PROGRESS = 0, RD_TASK_MAX_SPEED = 1,
       RD_TASK_N_STEP_PROGRESS = 2 /* agents B..D of the baselines' scenarios
                                      [REF baselines/scenarios/max_progress/austria.yml:16-18] */ };
/* observation outputs produced by rd_step/rd_reset */
enum {
  RD_OBS_LIDAR = 1,          /* f32 [N, n_beams] metres */
  RD_OBS_OCCUPANCY = 2,      /* u8 [N, 64, 64] 'lidar_occupancy' [REF dreamer/wrappers.py:372-414] */
  RD_OBS_LIDAR_NORM = 4,     /* lidar stored as r/15 - 0.5 [REF dreamer/tools.py:274] instead of metres */
  RD_OBS_LIDAR_F16 = 8,      /* lidar stored as IEEE half (round to nearest even of the float32 value): what Collect hands on at
                              * precision 16 [REF dreamer/wrappers.py:240-250 _convert; dreamer/dream.py:176-177].  lidar_dev then
                              * points to uint16 [N, n_beams]; halves the device->host bytes of the host-facing step.  The
                              * on-device policies read float32 scans and refuse this flag. */
  RD_OBS_NORM_BASELINES = 16 /* the model-free chain's NormalizeObservations: lidar, pose and velocity stored as
                              * (x - low) * (1 / (high - low)) per element, evaluated in float64 and rounded to float32
                              * (SinglePrecisionWrapper) [REF baselines/racing/environment/single_agent.py:66-99;
                              * baselines/racing/experiments/acme/experiment.py:66-75]; low/high = rd_config.obs_low/obs_high,
                              * the Box bounds of the env's observation space.  Excludes RD_OBS_LIDAR_NORM. */
};
enum { RD_NORM_LIDAR = 0, RD_NORM_POSE = 1, RD_NORM_VELOCITY = 2 };   /* index into rd_config.obs_low / obs_high */
/* action_repeat edge semantics [REF dreamer/wrappers.py:107-116 | baselines/.../single_agent.py:31-40] */
enum { RD_REPEAT_DREAMER = 0, RD_REPEAT_BASELINES = 1 };

/* state layout of rd_get_state / rd_set_state: f64 [RD_NF64][n_envs], i32 [RD_NI32][n_envs] (SoA).  Inside the library
 * the fields are kept as SoA of 16-byte groups (double2 pairs / one int4 + one int2 per env) so that every state access
 * of the step kernels is a 128-bit load or store; rd_get_state / rd_set_state convert. */
enum {
  RD_S_X = 0, RD_S_Y, RD_S_STEER, RD_S_V, RD_S_YAW, RD_S_YAWRATE, RD_S_SLIP,
  RD_S_TIME,       /* seconds since reset */
  RD_S_PROGRESS,   /* progress map value at the pose, [0,1] */
  RD_S_LAST,       /* lap + progress at the previous tick (reward bookkeeping) */
  RD_S_RETURN,     /* episode return so far */
  RD_S_START,      /* lap + progress at the last reset (episode progress = lap + progress - start) */
  RD_S_MAXPROG,    /* max over the episode's agent steps of lap + progress - 1, the per-episode statistic of tools.simulate
                    * [REF dreamer/tools.py:181,195]; -1 right after a reset (lap + progress - 1 is never negative) */
  RD_NF64
};
enum {
  RD_I_LAP = 0,     /* starts at 1 [REF dreamer/wrappers.py:218] */
  RD_I_CHECKPOINT,
  RD_I_FLAGS,       /* bit0 wrong_way, bit1 wall_collision, bit2 needs_reset, bit3 left_map, bit4 nan, bit5 opponent */
  RD_I_AGENT_STEP,  /* TimeLimit counter [REF dreamer/wrappers.py:147-154] */
  RD_I_EPISODE,     /* episodes started (reset-sampling counter) */
  RD_I_MAP,         /* map id of this env */
  RD_NI32
};
enum { RD_F_WRONG_WAY = 1, RD_F_COLLISION = 2, RD_F_NEEDS_RESET = 4, RD_F_LEFT_MAP = 8, RD_F_NAN = 16,
       RD_F_OPPONENT = 32 /* body overlaps another car of the same world (info['opponent_collisions'] non-empty) */ };

/* Single-track (bicycle) vehicle model parameters, SURVEY.md Appendix C [NEW-SPEC; in-tree anchors:
 * wheelbase 0.3302 REF ros_agent/agents/follow_the_gap/src/agent.py:78, max steering 0.42 and
 * max velocity 5.0 REF ros_agent/models/dreamer/racing_dreamer.py:14-16]. */
typedef struct rd_vehicle {
  double mu, c_sf, c_sr, lf, lr, h_cg, mass, inertia;
  double steer_min, steer_max, steer_vel_max; /* rad, rad/s */
  double v_switch, a_max, v_min, v_max;       /* CommonRoad acceleration constraint */
  double v_kinematic;                         /* |v| below this: kinematic model */
  double a_drive, a_brake, c_drag;            /* motor>=0: a = motor*a_drive - c_drag*v ; motor<0: braking */
  double steer_gain;                          /* steer target = steering * steer_gain * steer_max; default -1: a positive
                                               * steering action turns right [REF ros_agent/agents/dreamer/src/agent.py:111] */
  double body_length, body_width;             /* collision footprint (centred on the pose) */
} rd_vehicle;

typedef struct rd_config {
  int32_t abi_version;        /* = RD_ABI_VERSION */
  int32_t n_envs;
  int32_t n_beams;            /* 1080 [REF dreamer/dream.py:66] */
  int32_t action_repeat;      /* R [REF dreamer/dream.py:55, dreamer/wrappers.py:98-116] */
  int32_t repeat_semantics;   /* RD_REPEAT_* */
  int32_t obs_flags;          /* RD_OBS_* */
  int32_t task;               /* RD_TASK_* */
  int32_t laps;               /* done when lap > laps */
  int32_t terminate_on_collision;
  int32_t n_checkpoints;
  int32_t time_limit_steps;   /* TimeLimit wrapper, in agent steps; 0 = off [REF dreamer/wrappers.py:137-158] */
  int32_t auto_reset;         /* 1: a done env is reset inside the same step (obs = first obs of the new episode) */
  int32_t reset_mode;         /* RD_RESET_* used by auto-reset */
  int32_t rescale_actions;    /* 1: a' = (a+1)/2*(high-low)+low [REF dreamer/wrappers.py:129-134] */
  int32_t clip_actions;       /* 1: clip to [-1,1] first [REF baselines/racing/environment/single_agent.py:55-56] */
  int32_t progress_abs;       /* 1: reward uses |delta progress| */
  int64_t env_id_offset;      /* global id of env 0 (rank * n_envs for sharded runs): seeds differ per shard */
  uint64_t seed;
  double dt;                  /* 0.01 s sim tick [REF dreamer/callbacks.py:23] */
  double time_limit;          /* seconds [REF dreamer/scenarios/max_progress/austria.yml:10] */
  double collision_reward, progress_reward, frame_reward;
  double action_low[2], action_high[2]; /* [motor, steering] [REF dreamer/dream.py:138] */
  double lidar_fov;           /* rad, 270 deg [REF dreamer/tools.py:84-86] */
  double lidar_range_min, lidar_range_max; /* metres; 15 m [REF dreamer/tools.py:274] */
  double lidar_offset;        /* sensor position ahead of the pose along the heading, metres */
  float lidar_noise;          /* multiplicative U(1-a,1+a); 0 = off */
  float reserved0;
  /* ---- multi-agent worlds (SURVEY.md §8-f3) [REF baselines/scenarios/max_progress/austria.yml:3-34: four racecars
   *      A..D in one world; dreamer/dream.py:105-106 n_agents > 1; dreamer/wrappers.py:107-116,147-154 dict-of-agents
   *      step].  Env e is agent (e % agents_per_world) of world (e / agents_per_world); the agents of a world share its
   *      map, see each other in their LiDAR scans, collide with each other, stop repeating / time out / reset together
   *      (ActionRepeat: `not any(dones.values())` [REF wrappers.py:112]; tools.simulate: `if any(dones.values()):
   *      env.reset()` [REF dreamer/tools.py:178-179]).  agents_per_world <= 1: single-agent envs, fields below unused. */
  int32_t agents_per_world;   /* 1..RD_MAX_AGENTS; n_envs must be a multiple */
  int32_t agent_task[RD_MAX_AGENTS]; /* RD_TASK_* of agent index 0..3 (used when agents_per_world > 1) */
  int32_t n_step_progress;    /* n of n_step_progress, in sim ticks, 1..RD_MAX_NSTEP [REF .../austria.yml:18 n_steps: 10] */
  double ball_spacing;        /* random_ball / multi-agent random reset: metres of track between consecutive cars */
  /* ---- the model-free (baselines) wrapper chain ---- */
  int32_t time_limit_ticks;   /* gym TimeLimit(max_episode_steps) INSIDE ActionRepeat, i.e. counted in sim ticks: the tick
                               * that brings the episode's tick count to this value is done, subject to the repeat
                               * semantics like any task done [REF baselines/racing/experiments/acme/experiment.py:66-72;
                               * gym 0.18.0 wrappers/time_limit.py]; 0 = off */
  int32_t reserved1;
  double obs_low[3], obs_high[3]; /* RD_OBS_NORM_BASELINES: Box bounds of lidar / pose / velocity (RD_NORM_*) */
  rd_vehicle vehicle;
} rd_config;

/* Fills `cfg` with the defaults of the reference's dreamer training setup (action_repeat 4, laps 10, ...). */
void rd_default_config(rd_config* cfg);

/* Device pointers for one step's results.  Any pointer may be NULL = "do not produce".
 * [REF dreamer/wrappers.py:62-69 (obs dict + speed), :210-226 (Collect: f32 casts, progress, time)] */
typedef struct rd_outputs {
  float* lidar_dev;           /* [N, n_beams] float32 (IEEE half, i.e. uint16 storage, with RD_OBS_LIDAR_F16) */
  uint8_t* occupancy_dev;     /* [N, 64*64]   */
  float* pose_dev;            /* [N, 6] x,y,z,roll,pitch,yaw [REF dreamer/wrappers.py:395-401] */
  float* velocity_dev;        /* [N, 6] body-frame linear (vx,vy,0) + angular (0,0,yaw_rate) */
  float* speed_dev;           /* [N]   ||velocity[:3]|| ; 0 right after a reset [REF wrappers.py:66,74] */
  float* reward_dev;          /* [N]   summed over the repeated ticks [REF wrappers.py:110-116] */
  uint8_t* done_dev;          /* [N]   */
  float* progress_dev;        /* [N]   info['progress'] of the (possibly terminal) state */
  int32_t* lap_dev;           /* [N]   info['lap'] */
  float* time_dev;            /* [N]   info['time'] */
  uint8_t* flags_dev;         /* [N]   RD_F_* bits of the (possibly terminal) state */
  /* multi-agent worlds (NULL or left untouched when agents_per_world <= 1) */
  int32_t* rank_dev;          /* [N]   info['rank']: 1 = leader of the world by lap + progress (ties: lower agent index) */
  uint8_t* opponents_dev;     /* [N]   info['opponent_collisions'] as a bit mask over the world's agent indices */
  /* the two flags the reference's consumers read as booleans, ready-made (0 / 1) so that the host side decodes nothing
   * [REF baselines/racing/environment/tasks.py:8 info['wall_collision']; baselines/racing/experiments/sb3/
   * sb_experiment.py:82-88 info['wrong_way']] */
  uint8_t* wrong_way_dev;     /* [N]   info['wrong_way'] */
  uint8_t* wall_collision_dev;/* [N]   info['wall_collision'] */
} rd_outputs;

/* episode statistics accumulated on the device since the last rd_read_stats(reset=1)
 * [REF dreamer/tools.py:159-206 simulate(): per-episode return and max progress] */
typedef struct rd_stats {
  double episodes, return_sum, progress_sum, length_sum, collisions, laps_completed, env_steps, timeouts;
  double max_progress_sum;    /* sum over finished episodes of max_t (lap + progress - 1): what tools.simulate appends to
                               * max_progresses per episode [REF dreamer/tools.py:181,195] (progress_sum is the FINAL
                               * lap + progress - start instead); return_sum is its cum_reward [REF tools.py:182,194] */
} rd_stats;

/* ---- lifecycle: replaces RaceCarBaseEnv.__init__ -> MultiAgentScenario.from_spec + MultiAgentRaceEnv
 *      [REF dreamer/wrappers.py:10-16] ---- */
int rd_create(const rd_config* cfg, rd_env** out);
void rd_destroy(rd_env* env);
const char* rd_last_error(const rd_env* env_or_null);
int rd_abi_version(void);

/* ---- maps: replaces world._maps['occupancy'|'progress'|'obstacle'] = GridMap(np.load(maps.npz)[...])
 *      [REF dreamer/plotting/plot_trajectories.py:26-37; dreamer/wrappers.py:376]; all host pointers.
 *      bits: y-up rows of `row_words` u32, bit=1 drivable; dist: y-up u16 wavefront distance (cells);
 *      (col0,row0_yup): full-image cell index of the crop's lower-left cell; origin/resolution of the FULL image. */
int rd_upload_map(rd_env* env, int map_id, const uint32_t* bits_host, int h, int w, int row_words,
                  const uint16_t* dist_host, int dmax, double resolution, double origin_x, double origin_y,
                  int col0, int row0_yup, int full_h, const double* start_poses_host, int n_start,
                  const double* reset_poses_host, int n_reset);
/* map id per env (host int32[n_envs]); envs are grouped by map internally. */
int rd_assign_maps(rd_env* env, const int32_t* env_map_id_host);

/* ---- reset: replaces env.reset(mode=...) [REF dreamer/wrappers.py:71-77,91-92,156-158,410-414].
 *      mask_dev: u8[N] (NULL = all). Writes the reset observation of every env into `out`. ---- */
int rd_reset(rd_env* env, const uint8_t* mask_dev, int mode, const rd_outputs* out, void* stream);

/* ---- step: replaces Collect/TimeLimit/OccupancyMapObs/ReduceActionSpace/ActionRepeat/RaceCarWrapper.step
 *      -> MultiAgentRaceEnv.step [REF dreamer/wrappers.py:62-69,107-116,129-134,147-154,210-226,390-408].
 *      actions_dev: f32 [N,2] = [motor, steering] agent-facing ([-1,1] when rescale_actions). ---- */
int rd_step(rd_env* env, const float* actions_dev, const rd_outputs* out, void* stream);

/* ---- host-facing step: replaces `obs, reward, done, info = env.step(actions)` for callers whose actions and
 *      observations are HOST arrays (numpy), which is how the reference's driver loop calls the env
 *      [REF dreamer/tools.py:178-195 simulate()].  rd_host_init allocates, once, device result buffers and pinned
 *      host mirrors owned by the library and returns the HOST pointers in `host_out` (valid until rd_destroy).
 *      rd_step_host copies the actions in, steps the batch in `n_chunks` env-chunks pipelined over internal streams
 *      (chunk k's device->host copy overlaps chunk k+1's kernels) and returns when every result is in the host
 *      buffers.  Results are identical to rd_step's. ---- */
int rd_host_init(rd_env* env, int n_chunks, rd_outputs* host_out);
int rd_reset_host(rd_env* env, const uint8_t* mask_host, int mode);
int rd_step_host(rd_env* env, const float* actions_host);
/* Split form for callers that keep several env groups in flight (one handle per group, e.g. two half-batches whose policy
 * evaluations and copies overlap -- the asynchronous vector-env pattern): rd_step_host_begin copies the actions and
 * enqueues the whole step (kernels + device->host copies) without waiting, rd_step_host_end blocks until that step's
 * results are in the host buffers.  rd_step_host == begin + end.  One step may be pending per handle; the host buffers of
 * a handle must not be read between its begin and end. */
int rd_step_host_begin(rd_env* env, const float* actions_host);
int rd_step_host_end(rd_env* env);

/* ---- on-device policies (SURVEY.md §8-f2: policy-in-the-loop rollouts without a host round trip) ----
 * Follow-the-gap controller: replaces AgentNode.laserscan_callback + publish_drive_from_heading + PID.calculate
 * [REF ros_agent/agents/follow_the_gap/src/agent.py:128-193, 200-238, 45-55], one controller per env, state kept by
 * the handle and cleared whenever the env is reset (rd_reset, auto-reset inside rd_step).  The env's `lidar` row
 * (index 0 = left) is read in ROS order (index 0 = angle_min = -fov/2), i.e. reversed
 * [REF ros_agent/agents/dreamer/src/agent.py:65 np.flip]. */
typedef struct rd_gap_follower {
  /* controller constants [REF agent.py:73-104] */
  double lookahead;            /* 2 * max_speed^2 / (2 * max_decel) */
  double vehicle_width;        /* 0.3302 * 1.2 */
  double minimum_gap_length;   /* 0.2 m */
  double median_dev_threshold; /* 9.0 */
  double kp, ki, kd;           /* 1.4, 0.0, 0.1 */
  double max_vehicle_speed;    /* 6.0 */
  double max_steering_angle;   /* deg2rad(24) */
  double speed_limit_angle;    /* deg2rad(5) */
  double scan_dt;              /* seconds between scans = action_repeat * dt */
  /* scan geometry, derived the way the reference derives it from the LaserScan message */
  double angle_min, angle_increment, range_max;
  double pct_gamma;            /* np.percentile(q): fractional part of the virtual index */
  int32_t arc_first, arc_last; /* get_lidar_scan_arc(-90 deg, +90 deg) [REF agent.py:117-126], ROS order */
  int32_t filter_width;        /* int(deg2rad(10) / angle_increment) */
  int32_t pct_lo, pct_hi;      /* np.percentile(q): the two order statistics that are interpolated */
  int32_t reserved;
  /* drive command -> env action [NEW-SPEC: the reference publishes (steering_angle, speed) to a VESC]:
   * steering = steering_angle / (steer_gain * steer_max); motor = v*.c_drag/a_drive + speed_gain * (v* - v) with
   * v* = speed * speed_scale, both clipped to the sim-facing action range, then mapped back to the agent-facing
   * [-1, 1] when cfg.rescale_actions. */
  double speed_scale, speed_gain;
} rd_gap_follower;

/* Fills `g` with the reference node's constants and the geometry of `cfg`'s LiDAR. */
void rd_gap_follower_defaults(const rd_config* cfg, rd_gap_follower* g);
/* Allocates the per-env controller state (idempotent; replaces the parameters on a second call). */
int rd_policy_gap_follower_init(rd_env* env, const rd_gap_follower* g_or_null);
/* One controller update per env: lidar_dev f32 [N, n_beams] metres (an rd_step/rd_reset output), speed_dev f32 [N]
 * longitudinal speed or NULL (= the env's own state), actions_dev f32 [N,2] agent-facing (what rd_step takes),
 * debug_dev f64 [N,4] = (steering_angle, vehicle_speed, heading, heading_distance) or NULL. */
int rd_policy_gap_follower(rd_env* env, const float* lidar_dev, const float* speed_dev, float* actions_dev,
                           double* debug_dev, void* stream);
/* n_steps x (controller update -> rd_step) enqueued on `stream` with no host synchronisation; `out->lidar_dev` must
 * hold the current observation (rd_reset / previous rd_step with the same `out`).  The actions of the last step are
 * left in actions_dev (f32 [N,2], may be NULL). */
int rd_rollout_gap_follower(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, void* stream);

/* Dreamer agent: replaces RacingDreamer.action [REF ros_agent/models/dreamer/racing_dreamer.py:62-82] =
 * _preprocess_lidar -> RSSM.obs_step [REF ros_agent/models/dreamer/models.py:63-90] -> ActionDecoder(feat)
 * [REF models.py:307-346] -> SampleDist.mode() [REF ros_agent/helpers/tools.py:70-73], one agent per env, the recurrent
 * state (stoch, deter, previous action) kept by the handle and zeroed whenever the env is reset (`state is None`
 * [REF racing_dreamer.py:66-68]).  Every Dense / GRUCell is one launch of the tcgen05 kernel k_dense (TF32 tensor-core
 * products of hi/lo split float32 operands, float32 accumulation, csrc/rd_gemm.cuh).  Weights are HOST pointers in the checkpoint's own layout (Keras kernels
 * [in][out], the pickled `variables` of rssm.pkl / actor.pkl [REF ros_agent/helpers/tools.py:25-33]). */
typedef struct rd_dreamer_weights {
  int32_t stoch, deter, hidden, embed, actor_units, actor_layers;   /* 30, 200, 200, n_beams, 400, 4 */
  const float* gru_kernel;      /* [hidden][3*deter]  gates z | r | h  (tf.keras GRUCell, reset_after=True) */
  const float* gru_recurrent;   /* [deter][3*deter] */
  const float* gru_bias;        /* [2][3*deter]: input side, recurrent side */
  const float* img1_w; const float* img1_b;   /* [stoch+2][hidden], [hidden] */
  const float* obs1_w; const float* obs1_b;   /* [deter+embed][hidden], [hidden] */
  const float* obs2_w; const float* obs2_b;   /* [hidden][2*stoch], [2*stoch] */
  const float* actor_w[8]; const float* actor_b[8];   /* h0..h{L-1} then hout: [stoch+deter][units], [units][units].., [units][4] */
  const float* bn;              /* NULL ('tanh_normal') or [4][4] gamma, beta, moving_mean, moving_variance ('normalized_...') */
  float init_std, min_std, mean_scale, bn_eps;   /* 5, 1e-4, 5, 1e-3 */
  int32_t n_samples;            /* SampleDist samples: 100 */
  int32_t precision;            /* RD_PRECISION_* */
} rd_dreamer_weights;
/* arithmetic of the Dense / GRU products (accumulation is float32 either way) */
enum { RD_PRECISION_TF32X3 = 0,  /* hi/lo split operands, three tensor-core passes: float32-grade (the reference computes in float32) */
       RD_PRECISION_TF32 = 1     /* one TF32 pass (10-bit operand mantissas): ~1e-3 relative per layer, fastest */ };
/* noise: where the standard-normal draws of the posterior sample and of SampleDist come from */
enum { RD_NOISE_ZERO = 0,      /* none: stoch = mean, action = tanh(actor mean)  [NEW-SPEC, deterministic evaluation] */
       RD_NOISE_PHILOX = 1,    /* Philox(cfg.seed; env id, policy step)          [NEW-SPEC, the reference uses TF's RNG] */
       RD_NOISE_EXPLICIT = 2   /* caller-provided draws (teacher-forced parity tests) */ };
#define RD_DREAMER_DEBUG_FLOATS 68   /* per env: posterior mean[30] std[30] | actor mean[2] std[2] action[2] log_prob index */
/* Allocates the weights and the per-env latent state and packs the weights on the device (K-major TF32 operands, the
 * packing rd_policy_dreamer_set_weights uses); returns after the packing finished.  The scans are normalised on the
 * device (x/15 - 0.5) unless the env emits normalised ones.  Idempotent: a second call replaces the agent and clears the
 * state; a rejected call (RD_ERR_INVALID, e.g. a device pointer in w) leaves the current agent working. */
int rd_policy_dreamer_init(rd_env* env, const rd_dreamer_weights* w);
/* One agent step per env.  lidar_dev f32 [N, n_beams] (an rd_step / rd_reset output), actions_dev f32 [N,2]
 * agent-facing (what rd_step takes; its rescale is postprocess_action [REF racing_dreamer.py:54-60]).
 * eps_stoch_dev f32 [N,30] and eps_actor_dev f32 [N, n_samples, 2] are read when noise == RD_NOISE_EXPLICIT.
 * debug_dev: NULL or f32 [N*60] posterior (mean|std) followed by [N*8] actor diagnostics. */
int rd_policy_dreamer(rd_env* env, const float* lidar_dev, float* actions_dev, int noise, const float* eps_stoch_dev,
                      const float* eps_actor_dev, float* debug_dev, void* stream);
/* latent state access: stoch f32 [N,30], deter f32 [N,deter], action f32 [N,2] (any may be NULL) */
int rd_policy_dreamer_get_state(rd_env* env, float* stoch_dev, float* deter_dev, float* action_dev, void* stream);
int rd_policy_dreamer_set_state(rd_env* env, const float* stoch_dev, const float* deter_dev, const float* action_dev,
                                void* stream);
/* n_steps x (agent step -> rd_step) enqueued on `stream` with no host synchronisation (see rd_rollout_gap_follower). */
int rd_rollout_dreamer(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, int noise, void* stream);

/* Training mode: Dreamer.policy(obs, state, training=True) [REF dreamer/dreamer.py, Dreamer.policy, _exploration].
 * The head takes ONE sample of the actor distribution, a = tanh(mean + sd e1), and explores:
 * a' = clip(a + amount_k e2, -1, 1) in float32, one rounding per operation.  a' is written to actions_dev and kept in
 * the latent state as the previous action.  amount_k = expl amount * 0.5^(env_steps / decay) (decay > 0), at least
 * min_amount (min_amount > 0), computed in float64 and rounded once to float32; env_steps then advances by
 * n_envs * action_repeat (evaluation steps leave it).  noise: RD_NOISE_PHILOX draws (e1, e2) from one Philox block,
 * counter (env id, agent step, 0, tag), key (seed_lo, seed_hi ^ tag), apart from the evaluation-mode and posterior
 * streams; RD_NOISE_ZERO: e1 = e2 = 0; RD_NOISE_EXPLICIT reads eps_stoch_dev f32 [N,30], eps_sample_dev f32 [N,2] (e1)
 * and eps_expl_dev f32 [N,2] (e2).  debug_dev as rd_policy_dreamer's; its action is a (before exploration), its
 * log_prob that of a, its index 0. */
typedef struct rd_dreamer_exploration {
  double amount;              /* expl_amount: 0.3 */
  double decay;               /* expl_decay: 0 = constant amount */
  double min_amount;          /* expl_min: 0 = no floor */
  int64_t env_steps;          /* the schedule's env-step counter */
} rd_dreamer_exploration;
/* rd_policy_dreamer_init sets env_steps to 0 and leaves the rest (0.3, 0, 0 until set). */
int rd_policy_dreamer_set_exploration(rd_env* env, const rd_dreamer_exploration* x);
int rd_policy_dreamer_get_exploration(rd_env* env, rd_dreamer_exploration* x);
int rd_policy_dreamer_train(rd_env* env, const float* lidar_dev, float* actions_dev, int noise, const float* eps_stoch_dev,
                            const float* eps_sample_dev, const float* eps_expl_dev, float* debug_dev, void* stream);
/* n_steps x (training agent step -> rd_step) enqueued on `stream`, no host synchronisation. */
int rd_rollout_dreamer_train(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, int noise, void* stream);
/* New weights for an initialised agent, packed on the device on `stream` into the buffers rd_policy_dreamer_init
 * allocated, bit for bit as init packs them.  w: the layout rd_policy_dreamer_init takes, its array pointers DEVICE
 * memory of the env's device (on_device = 1, e.g. a learner's tensors) or host memory (on_device = 0: copied with
 * cudaMemcpyAsync on `stream` through a staging buffer the handle owns).  No allocation; the latent state, the Philox
 * step counter and the exploration state are kept.  Steps enqueued on `stream` before the call use the old weights,
 * the ones after it the new ones.  The architecture, BN presence, precision and head scalars must equal the init's
 * (else RD_ERR_INVALID and nothing changes). */
int rd_policy_dreamer_set_weights(rd_env* env, const rd_dreamer_weights* w, int on_device, void* stream);

/* Dreamer agent on 'lidar_occupancy' observations [REF dreamer/dream.py:64-66]: the image encoder ConvEncoder
 * [UPSTREAM-RECALL: danijar Dreamer models.py ConvEncoder] replaces _preprocess_lidar in front of the same RSSM and actor.
 * The u8 image [N,64,64] is cast to float (no scaling), then four Conv2D(kernel 4, stride 2, 'valid', relu) layers with
 * depth, 2 depth, 4 depth, 8 depth filters (31x31, 14x14, 6x6, 2x2 outputs); the 2x2x(8 depth) output flattened in
 * (y, x, c) order is the embed (32 depth floats) obs1 reads.  conv1 runs on CUDA cores, conv2..conv4 as implicit GEMMs
 * on the k_dense tensor-core kernel (csrc/rd_gemm.cuh).  Only depth 32 (the reference's cnn_depth) is accepted. */
typedef struct rd_dreamer_conv_encoder {
  int32_t depth;              /* cnn_depth: 32 */
  const float* w[4];          /* Keras Conv2D kernels [4][4][Cin][Cout], Cin = 1, d, 2d, 4d; Cout = d, 2d, 4d, 8d */
  const float* b[4];          /* [Cout] */
} rd_dreamer_conv_encoder;
/* As rd_policy_dreamer_init, for an encoder agent: w->embed = 32 * enc->depth (obs1_w [deter + embed][hidden]); the env
 * must produce occupancy (RD_OBS_OCCUPANCY).  Allocates the encoder's activations (~0.4 MB per env in tf32x3).  Re-init
 * with either init replaces the agent; a rejected call leaves the current one working. */
int rd_policy_dreamer_init_occupancy(rd_env* env, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc);
/* rd_policy_dreamer / rd_policy_dreamer_train for an encoder agent: occupancy_dev u8 [N,64,64] (an rd_step output). */
int rd_policy_dreamer_occupancy(rd_env* env, const uint8_t* occupancy_dev, float* actions_dev, int noise,
                                const float* eps_stoch_dev, const float* eps_actor_dev, float* debug_dev, void* stream);
int rd_policy_dreamer_occupancy_train(rd_env* env, const uint8_t* occupancy_dev, float* actions_dev, int noise,
                                      const float* eps_stoch_dev, const float* eps_sample_dev, const float* eps_expl_dev,
                                      float* debug_dev, void* stream);
/* rd_policy_dreamer_set_weights for an encoder agent: the encoder's arrays follow the same on_device rule. */
int rd_policy_dreamer_set_weights_occupancy(rd_env* env, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc,
                                            int on_device, void* stream);
/* The encoder stage alone: embed_dev f32 [N][32 depth] = hi + lo of what obs1 reads.  The latent state is untouched. */
int rd_dreamer_encode_occupancy(rd_env* env, const uint8_t* occupancy_dev, float* embed_dev, void* stream);
/* rd_rollout_dreamer, rd_rollout_dreamer_train, rd_rollout_store (RD_STORE_POLICY_DREAMER*), get/set_state and the
 * per-env state zeroing serve both agent kinds; an encoder agent's rollout reads out->occupancy_dev.  The lidar entry
 * points fail for an encoder agent and the occupancy ones for a lidar agent (RD_ERR_INVALID). */

/* ---- several Dreamer agents in one env batch: env e is driven by agent agent_of_env[e].  Replaces the reference's ways
 *      of running more than one checkpoint: one agent per car of a multi-agent scenario
 *      [REF baselines/scenarios/max_progress/austria.yml:3-34 (cars A..D, each with its own agent)], the evaluation of
 *      several checkpoints [REF dreamer/evaluations/run_evaluation.py:43-94 (a loop over checkpoints and tracks)], and
 *      Dreamer._exploration per learner [REF dreamer/dreamer.py, Dreamer._exploration].
 *      Env e's actions, state rows, debug rows and Philox draws are bit for bit what the single-agent policy with agent
 *      agent_of_env[e]'s weights gives env e on the same batch: the draws stay keyed by the env id.  Internally the rows
 *      are ordered by agent, each agent's from a multiple of 128 (csrc/rd_dreamer.cuh); every entry point keeps env order.
 *      rd_policy_dreamer[_train], _occupancy[_train], rd_rollout_dreamer[_train], rd_rollout_store (both Dreamer
 *      policies), get/set_state, rd_dreamer_encode_occupancy and the per-env state zeroing serve a multi-agent policy
 *      unchanged.  On a policy with more than one agent, rd_policy_dreamer_set_weights[_occupancy] and
 *      rd_policy_dreamer_set/get_exploration return RD_ERR_INVALID: use the per-agent calls below. ---- */
#define RD_MAX_DREAMER_AGENTS 8
/* n_agents = G in 1..RD_MAX_DREAMER_AGENTS; w[G]; enc: NULL (lidar agents, as rd_policy_dreamer_init) or enc[G]
 * (ConvEncoder agents, as rd_policy_dreamer_init_occupancy); agent_of_env_host int32 [N] host values in [0, G), every
 * agent owning at least one env, in any arrangement.  Every agent has agent 0's architecture, precision, n_samples,
 * head scalars and encoder depth; BN presence may differ per agent.  Otherwise, and for everything
 * rd_policy_dreamer_init rejects, RD_ERR_INVALID and the current agent keeps working.  Replaces the current agent(s),
 * zeroes the state and every agent's env_steps, and returns after the packing finished.  G = 1 is
 * rd_policy_dreamer_init[_occupancy]. */
int rd_policy_dreamer_init_agents(rd_env* env, int32_t n_agents, const rd_dreamer_weights* w,
                                  const rd_dreamer_conv_encoder* enc, const int32_t* agent_of_env_host);
/* rd_policy_dreamer_set_weights[_occupancy] for agent `agent` (enc: NULL for lidar agents): packs that agent's weights
 * on `stream` with no allocation; the other agents' weights and every env's latent state are untouched.  The agent's
 * BN presence must be the one it was initialised with. */
int rd_policy_dreamer_set_agent_weights(rd_env* env, int32_t agent, const rd_dreamer_weights* w,
                                        const rd_dreamer_conv_encoder* enc, int on_device, void* stream);
/* rd_policy_dreamer_set/get_exploration for agent `agent`.  A training step advances the agent's env_steps by
 * (its envs) x action_repeat, Dreamer's len(reset) x action_repeat over the envs it drives. */
int rd_policy_dreamer_set_agent_exploration(rd_env* env, int32_t agent, const rd_dreamer_exploration* x);
int rd_policy_dreamer_get_agent_exploration(rd_env* env, int32_t agent, rd_dreamer_exploration* x);

/* ---- feed-forward Gaussian actor (the model-free baselines' actors, e.g. SB3's SAC and PPO policies): a trunk of
 *      1..RD_MLP_MAX_LAYERS Linear + activation layers over the env's scan, then a head of two action means and two
 *      log standard deviations.  The trunk and head products run on the tcgen05 tensor cores in three TF32 passes over
 *      hi/lo split operands (float32-grade).  The actor reads the baselines chain's observation, the flattened scan
 *      normalised to [0, 1]: init needs RD_OBS_NORM_BASELINES, float32 lidar without occupancy, clip_actions = 1 and
 *      rescale_actions = 0 (RD_ERR_INVALID otherwise).  One actor per handle, stateless per env. ---- */
#define RD_MLP_MAX_LAYERS 4
#define RD_MLP_MAX_WIDTH 1024
#define RD_MLP_DEBUG_FLOATS 4   /* per env: mean[2] std[2] of the Gaussian before the squash */
enum { RD_ACT_RELU = 0, RD_ACT_TANH = 1 };
enum { RD_HEAD_SQUASHED = 0, /* per-state log_std layer clamped to [log_std_min, log_std_max]; a = tanh(mean + std e) */
       RD_HEAD_DIAG = 1      /* state-independent log_std vector [2]; a = mean + std e, unclipped */ };
typedef struct rd_mlp_actor {
  int32_t n_layers;             /* trunk layers, 1..RD_MLP_MAX_LAYERS */
  int32_t in_features;          /* = cfg.n_beams */
  int32_t width[RD_MLP_MAX_LAYERS];   /* output width of each trunk layer, 1..RD_MLP_MAX_WIDTH */
  int32_t activation;           /* RD_ACT_* after every trunk layer */
  int32_t head;                 /* RD_HEAD_* */
  float log_std_min, log_std_max;     /* RD_HEAD_SQUASHED clamp */
  /* PyTorch layout (nn.Linear): weight [out][in], bias [out]; host pointers, or device pointers with on_device */
  const float* w[RD_MLP_MAX_LAYERS];
  const float* b[RD_MLP_MAX_LAYERS];
  const float* mean_w;          /* [2][width[n_layers - 1]] */
  const float* mean_b;          /* [2] */
  const float* log_std_w;       /* RD_HEAD_SQUASHED: [2][width[n_layers - 1]]; else ignored */
  const float* log_std_b;       /* RD_HEAD_SQUASHED: [2]; else ignored */
  const float* log_std;         /* RD_HEAD_DIAG: [2]; else ignored */
} rd_mlp_actor;
/* Packs the actor's weights (host pointers) for the handle's envs; replaces an earlier actor.  Every check (the env
 * config above, the architecture, the pointers) runs before any device work: a rejected init changes nothing. */
int rd_policy_mlp_init(rd_env* env, const rd_mlp_actor* a);
/* One actor step for every env: obs_dev f32 [N, n_beams] (the env's lidar output) -> actions_dev f32 [N, 2], the
 * agent-facing action rd_step reads.  deterministic: e = 0 (SAC: tanh(mean); PPO: mean); else e ~ N(0, 1) per noise mode
 * (RD_NOISE_PHILOX: block (env id, step, 0, stream tag) of Philox4x32-10 keyed (seed_lo, seed_hi ^ tag), Box-Muller
 * normals z0, z1; RD_NOISE_ZERO: e = 0; RD_NOISE_EXPLICIT: eps_dev f32 [N, 2]).  debug_dev (may be NULL) f32
 * [N, RD_MLP_DEBUG_FLOATS].  The step counter advances by one per call. */
int rd_policy_mlp(rd_env* env, const float* obs_dev, float* actions_dev, int deterministic, int noise, const float* eps_dev,
                  float* debug_dev, void* stream);
/* New weights of the init's architecture (n_layers, widths, in_features, activation, head, clamp bounds; else
 * RD_ERR_INVALID and nothing changes), packed on `stream` by init's packer.  on_device: the pointers are device memory
 * of the handle's device, read on `stream` without a host synchronisation.  The step counter is kept. */
int rd_policy_mlp_set_weights(rd_env* env, const rd_mlp_actor* w, int on_device, void* stream);
/* n_steps x (rd_policy_mlp on out->lidar_dev -> rd_step); noise RD_NOISE_PHILOX or RD_NOISE_ZERO; the actions of the
 * last step are left in actions_dev (may be NULL). */
int rd_rollout_mlp(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, int deterministic, int noise,
                   void* stream);
/* Uniform random actions, any env config: per env and call, Philox4x32-10 block (env id, step, 0, stream tag) keyed
 * (seed_lo, seed_hi ^ tag), a_k = 2 (x_k >> 8) 2^-24 - 1 in [-1, 1) for k = 0, 1 (exact in float32).  The handle's
 * random-action step counter advances by one per call. */
int rd_policy_random(rd_env* env, float* actions_dev, void* stream);
/* n_steps x (rd_policy_random -> rd_step); actions_dev as rd_rollout_mlp */
int rd_rollout_random(rd_env* env, int n_steps, const rd_outputs* out, float* actions_dev, void* stream);

/* ---- device-resident episode store (SURVEY.md §8-f1): records the Collect rows of every env's episodes on the device
 *      [REF dreamer/wrappers.py:198-250], exactly the episodes episodes.EpisodeRecorder hands to its callbacks, and
 *      samples fixed-length chunks the way tools.load_episodes does [REF dreamer/tools.py:235-264].  The env must have
 *      auto_reset = 0: the store resets the envs whose episode ended, after recording the terminal row.
 *      Storage: a ring of capacity_rows rows per env (memory n_envs x capacity_rows x row bytes); an env's oldest
 *      committed episodes are evicted as its ring wraps.  capacity_rows must exceed the longest episode the config
 *      allows (time_limit_steps, time_limit_ticks / action_repeat, the task's time_limit / (dt * action_repeat)). ---- */
enum { RD_STORE_LIDAR = 1, RD_STORE_POSE = 2, RD_STORE_VELOCITY = 4, RD_STORE_SPEED = 8,
       RD_STORE_OCCUPANCY = 16 /* 'lidar_occupancy', u8 [64,64,1]; needs RD_OBS_OCCUPANCY */ };   /* keep_obs bits */
enum { RD_STORE_POLICY_GAP_FOLLOWER = 0, RD_STORE_POLICY_DREAMER = 1,
       RD_STORE_POLICY_DREAMER_TRAIN = 2, /* rd_rollout_dreamer_train's agent step */
       RD_STORE_POLICY_MLP = 3,           /* rd_rollout_mlp, deterministic actions */
       RD_STORE_POLICY_MLP_TRAIN = 4,     /* rd_rollout_mlp, sampled actions (noise RD_NOISE_PHILOX or RD_NOISE_ZERO) */
       RD_STORE_POLICY_RANDOM = 5         /* rd_rollout_random */ };                                  /* rd_rollout_store */
typedef struct rd_store_config {
  int32_t capacity_rows;      /* rows per env */
  int32_t precision;          /* 32 | 16: float keys as float32 | IEEE half [REF dreamer/wrappers.py:240-250 _convert] */
  int32_t keep_obs;           /* RD_STORE_* observation keys to store (action, reward, discount, progress, time always) */
  int32_t reset_mode;         /* RD_RESET_* of the resets of finished envs; -1 = cfg.reset_mode */
  uint64_t seed;              /* sampler: Philox key (seed_lo, seed_hi ^ stream tag) */
} rd_store_config;
/* A sampled batch: caller-owned device buffers [B, L, ...] in the store's precision; NULL = not produced. */
typedef struct rd_store_batch {
  void* lidar_dev;            /* [B, L, n_beams] */
  uint8_t* occupancy_dev;     /* [B, L, 64*64]   */
  void* pose_dev;             /* [B, L, 6] */
  void* velocity_dev;         /* [B, L, 6] */
  void* speed_dev;            /* [B, L] */
  void* action_dev;           /* [B, L, 2] */
  void* reward_dev;           /* [B, L] */
  void* discount_dev;         /* [B, L] */
  void* progress_dev;         /* [B, L] */
  void* time_dev;             /* [B, L] */
  int64_t* episode_id_dev;    /* [B] id of the chunk's episode, -1 = no chunk (zero rows) */
  int32_t* start_dev;         /* [B] first row of the chunk in its episode, -1 = no chunk */
} rd_store_batch;
typedef struct rd_store_summary {
  int64_t committed;          /* episodes committed since rd_store_init (the next episode id) */
  int64_t held;               /* episodes held (committed and not evicted) */
  int64_t held_rows;          /* rows of the held episodes */
  int64_t evicted;            /* committed - held */
  int64_t invalid_requests;   /* caller-given sample indices that named no held chunk */
  int64_t draws;              /* drawing rd_store_sample calls so far (the counter k of the draw law) */
  int64_t capacity_rows, max_episode_steps;
} rd_store_summary;
typedef struct rd_store_episode { int64_t id, env, length; } rd_store_episode;

/* Allocates the store of the handle (replaces an existing one). */
int rd_store_init(rd_env* env, const rd_store_config* sc);
/* rd_reset of every env + the first row of each env's new episode (episodes in progress are dropped, held ones kept). */
int rd_store_reset(rd_env* env, const rd_outputs* out, void* stream);
/* rd_step -> record every env's row -> commit the episodes of the worlds with a done car (ids in env order) -> reset
 * exactly those envs (the others are not observed again) -> record their first rows.  Afterwards `out` holds, for reset
 * envs, the first observation of the next episode, with reward and done of the finished step.  No host synchronisation.
 * out must provide lidar (if stored), occupancy (if stored), pose, velocity, speed, reward, done, progress, lap, time. */
int rd_store_step(rd_env* env, const float* actions_dev, const rd_outputs* out, void* stream);
/* n_steps x (policy -> rd_store_step); policy RD_STORE_POLICY_*, noise as rd_rollout_dreamer (ignored for the gap
 * follower); the actions of the last step are left in actions_dev (may be NULL). */
int rd_rollout_store(rd_env* env, int policy, int n_steps, const rd_outputs* out, float* actions_dev, int noise,
                     void* stream);
/* batch chunks of `length` rows.  ids_dev == NULL: drawn over the held episodes of at least length + 1 rows in commit
 * order (draw law in csrc/rd_store.cuh; balance: the reference's balance=True start).  Else ids_dev i64 [B] and
 * starts_dev i32 [B] name the chunks; they are checked on the device, and must not overlap the episode_id / start
 * outputs (RD_ERR_INVALID).  Asynchronous. */
int rd_store_sample(rd_env* env, int batch, int length, int balance, const int64_t* ids_dev, const int32_t* starts_dev,
                    const rd_store_batch* out, void* stream);
/* Synchronises `stream`.  episodes_host (may be NULL): the first max_episodes held episodes in commit order. */
int rd_store_info(rd_env* env, rd_store_summary* out_host, rd_store_episode* episodes_host, int64_t max_episodes,
                  void* stream);

/* ---- import arena: episodes from outside the store (saved files, other runs) sampled together with the recorded ones.
 *      One ring of import_capacity_rows rows per key, same row format and precision as the env rings; imported
 *      episode k (0, 1, ... in import order since rd_store_import_init) has id RD_STORE_IMPORTED_ID0 + k and env -1.
 *      It is held while its first row has not been overwritten, so importing past the arena's end evicts the oldest
 *      imported episodes.  Draws of rd_store_sample pick from one list: the held imported episodes in import order, then
 *      the held recorded episodes in commit order.  Imports never touch the env rings or the recorded episodes;
 *      rd_store_reset keeps imported episodes, rd_store_init drops them. ---- */
#define RD_STORE_IMPORTED_ID0 (INT64_C(1) << 62)
enum { RD_STORE_U8 = 1, RD_STORE_F16 = 2, RD_STORE_F32 = 4, RD_STORE_F64 = 8 };   /* staged element type (= its bytes) */
/* Staged rows of the episodes of one rd_store_import call, back to back: caller-owned device buffers [rows, ...] in the
 * row shapes of rd_store_batch; a kept key needs its pointer and type (float keys F16 | F32 | F64, occupancy U8),
 * others are ignored.  Floats are rounded once to the store's precision (numpy astype). */
typedef struct rd_store_import_rows {
  const void* lidar_dev; const void* occupancy_dev; const void* pose_dev; const void* velocity_dev; const void* speed_dev;
  const void* action_dev; const void* reward_dev; const void* discount_dev; const void* progress_dev; const void* time_dev;
  int32_t lidar_type, occupancy_type, pose_type, velocity_type, speed_type, action_type, reward_type, discount_type,
          progress_type, time_type;
} rd_store_import_rows;
typedef struct rd_store_import_summary {
  int64_t imported;           /* episodes imported since rd_store_import_init (the next imported id - ID0) */
  int64_t held;               /* imported episodes held */
  int64_t held_rows;          /* rows of the held imported episodes */
  int64_t evicted;            /* imported - held */
  int64_t capacity_rows;      /* arena rows (0: no arena) */
} rd_store_import_summary;

/* Allocates the import arena of the store (after rd_store_init; replaces an existing arena and its episodes). */
int rd_store_import_init(rd_env* env, int32_t import_capacity_rows);
/* Imports n_episodes episodes of lengths_host[i] rows (1 <= length <= import_capacity_rows), staged in `rows`.  rows ==
 * NULL counts them as imported and at once overwritten (ids and arena rows advance, nothing is held or read): for the
 * episodes a caller knows later imports overwrite.  Asynchronous; the staged buffers must stay valid until the work
 * enqueued on `stream` has run. */
int rd_store_import(rd_env* env, int32_t n_episodes, const int32_t* lengths_host, const rd_store_import_rows* rows,
                    void* stream);
/* Synchronises `stream`.  episodes_host (may be NULL): the first max_episodes held imported episodes in import order. */
int rd_store_import_info(rd_env* env, rd_store_import_summary* out_host, rd_store_episode* episodes_host,
                         int64_t max_episodes, void* stream);

/* ---- stage entry points (teacher-forced parity tests; each is one kernel of the step) ---- */
/* a2 LiDAR [REF dreamer/scenarios/max_progress/austria.yml:7 'lidar' sensor]: poses f64 [n,3]=(x,y,yaw),
 * map_ids i32[n] sorted ascending or NULL (= map 0), ranges f32 [n, n_beams].  With agents_per_world = A > 1 consecutive
 * poses form worlds (n must be a multiple of A, the cars of a world on one map) and see each other. */
int rd_lidar_cast(rd_env* env, const double* poses_dev, const int32_t* map_ids_host, int n,
                  float* ranges_dev, void* stream);
/* a5 OccupancyMapObs.step [REF dreamer/wrappers.py:390-408]: poses f64 [n,3], out u8 [n,64*64]. */
int rd_occupancy_obs(rd_env* env, const double* poses_dev, const int32_t* map_ids_host, int n,
                     uint8_t* out_dev, void* stream);
/* a1 dynamics only: state f64 [7][n] SoA (x,y,steer,v,yaw,yaw_rate,slip) in/out,
 * commands f64 [n,2] = sim-facing (motor, steering), n_ticks ticks of cfg.dt. */
int rd_dynamics(rd_env* env, double* state_dev, const double* commands_dev, int n, int n_ticks, void* stream);

/* a7/a8 one sim tick of progress / lap / wrong-way bookkeeping + task reward / done for teacher-forced poses (single-car
 * rule, cfg.task) [REF consumers: dreamer/wrappers.py:218-219; dreamer/tools.py:195; baselines/racing/environment/
 * tasks.py:4-22; task parameters dreamer/scenarios/max_progress/austria.yml:8-10]:
 *   kin_dev      f64 [5][n] SoA (x, y, yaw, v, slip): the car AFTER the tick
 *   steering_dev f64 [n] sim-facing steering command (max_speed reward) or NULL (= 0)
 *   map_ids_host as rd_lidar_cast
 *   book_f64_dev f64 [3][n] (time, progress, last = lap + progress of the previous tick), in/out
 *   book_i32_dev i32 [3][n] (lap, checkpoint, flags), in/out
 *   reward_dev   f64 [n] the tick's reward;  done_dev u8 [n] the task's done (no ActionRepeat / TimeLimit on top) */
int rd_reward_done(rd_env* env, const double* kin_dev, const double* steering_dev, const int32_t* map_ids_host, int n,
                   double* book_f64_dev, int32_t* book_i32_dev, double* reward_dev, uint8_t* done_dev, void* stream);

/* ---- state access (checkpoint/resume; teacher forcing); either pointer may be NULL.  The ring of the n_step_progress
 *      task is not part of the layout: restoring the float64 part restarts it from the restored lap + progress ---- */
int rd_get_state(rd_env* env, double* f64_dev, int32_t* i32_dev, void* stream);
int rd_set_state(rd_env* env, const double* f64_dev, const int32_t* i32_dev, void* stream);

/* ---- episode statistics (K5): device-side accumulators -> host struct (synchronises `stream`) ---- */
int rd_read_stats(rd_env* env, rd_stats* out_host, int reset, void* stream);

/* ---- introspection for bench/profiling ---- */
/* kernels launched by this handle so far */
int64_t rd_launch_count(const rd_env* env);
/* per-kernel device time: when enabled, every launch is bracketed by CUDA events on its stream;
 * rd_read_timing synchronises those events and returns the accumulated milliseconds per kernel class. */
typedef struct rd_timing {
  double step_ms, lidar_ms, occupancy_ms, reset_ms;
  int64_t step_launches, lidar_launches, occupancy_launches, reset_launches;
  double policy_ms;
  int64_t policy_launches;
} rd_timing;
int rd_enable_timing(rd_env* env, int enable);
int rd_read_timing(rd_env* env, rd_timing* out_host, int reset);

#ifdef __cplusplus
}
#endif
#endif /* RD_ENV_H */
