"""ctypes mirror of include/rd_env.h and the loader of librd_env.so.

The loader fails loudly: there is no CPU or PyTorch fallback for the env step.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

ABI_VERSION = 3
MAX_AGENTS = 4   # RD_MAX_AGENTS
MAX_NSTEP = 32   # RD_MAX_NSTEP

# enums (include/rd_env.h)
RESET_GRID, RESET_RANDOM, RESET_RANDOM_BIDIRECTIONAL, RESET_RANDOM_BALL = 0, 1, 2, 3
RESET_MODES = {"grid": RESET_GRID, "random": RESET_RANDOM, "random_bidirectional": RESET_RANDOM_BIDIRECTIONAL,
               "random_ball": RESET_RANDOM_BALL}
TASK_MAX_PROGRESS, TASK_MAX_SPEED, TASK_N_STEP_PROGRESS = 0, 1, 2
TASKS = {"maximize_progress": TASK_MAX_PROGRESS, "max_progress": TASK_MAX_PROGRESS,
         "max_speed": TASK_MAX_SPEED, "maximize_speed": TASK_MAX_SPEED, "n_step_progress": TASK_N_STEP_PROGRESS}
OBS_LIDAR, OBS_OCCUPANCY, OBS_LIDAR_NORM, OBS_LIDAR_F16, OBS_NORM_BASELINES = 1, 2, 4, 8, 16
NORM_LIDAR, NORM_POSE, NORM_VELOCITY = 0, 1, 2
REPEAT_DREAMER, REPEAT_BASELINES = 0, 1

S_X, S_Y, S_STEER, S_V, S_YAW, S_YAWRATE, S_SLIP, S_TIME, S_PROGRESS, S_LAST, S_RETURN, S_START, S_MAXPROG, NF64 = range(14)
I_LAP, I_CHECKPOINT, I_FLAGS, I_AGENT_STEP, I_EPISODE, I_MAP, NI32 = range(7)
F_WRONG_WAY, F_COLLISION, F_NEEDS_RESET, F_LEFT_MAP, F_NAN, F_OPPONENT = 1, 2, 4, 8, 16, 32


class RdVehicle(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "mu", "c_sf", "c_sr", "lf", "lr", "h_cg", "mass", "inertia",
        "steer_min", "steer_max", "steer_vel_max",
        "v_switch", "a_max", "v_min", "v_max",
        "v_kinematic",
        "a_drive", "a_brake", "c_drag",
        "steer_gain",
        "body_length", "body_width")]


class RdConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("n_envs", C.c_int32), ("n_beams", C.c_int32), ("action_repeat", C.c_int32),
        ("repeat_semantics", C.c_int32), ("obs_flags", C.c_int32), ("task", C.c_int32), ("laps", C.c_int32),
        ("terminate_on_collision", C.c_int32), ("n_checkpoints", C.c_int32), ("time_limit_steps", C.c_int32),
        ("auto_reset", C.c_int32), ("reset_mode", C.c_int32), ("rescale_actions", C.c_int32),
        ("clip_actions", C.c_int32), ("progress_abs", C.c_int32),
        ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("dt", C.c_double), ("time_limit", C.c_double),
        ("collision_reward", C.c_double), ("progress_reward", C.c_double), ("frame_reward", C.c_double),
        ("action_low", C.c_double * 2), ("action_high", C.c_double * 2),
        ("lidar_fov", C.c_double), ("lidar_range_min", C.c_double), ("lidar_range_max", C.c_double),
        ("lidar_offset", C.c_double),
        ("lidar_noise", C.c_float), ("reserved0", C.c_float),
        ("agents_per_world", C.c_int32), ("agent_task", C.c_int32 * MAX_AGENTS), ("n_step_progress", C.c_int32),
        ("ball_spacing", C.c_double),
        ("time_limit_ticks", C.c_int32), ("reserved1", C.c_int32),
        ("obs_low", C.c_double * 3), ("obs_high", C.c_double * 3),
        ("vehicle", RdVehicle),
    ]

    def copy(self) -> "RdConfig":
        out = RdConfig()
        C.memmove(C.byref(out), C.byref(self), C.sizeof(RdConfig))
        return out


class RdOutputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "lidar_dev", "occupancy_dev", "pose_dev", "velocity_dev", "speed_dev", "reward_dev", "done_dev",
        "progress_dev", "lap_dev", "time_dev", "flags_dev", "rank_dev", "opponents_dev", "wrong_way_dev",
        "wall_collision_dev")]


class RdStats(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "episodes", "return_sum", "progress_sum", "length_sum", "collisions", "laps_completed", "env_steps",
        "timeouts", "max_progress_sum")]

    def as_dict(self):
        return {n: float(getattr(self, n)) for n, _ in self._fields_}


class RdTiming(C.Structure):
    _fields_ = [("step_ms", C.c_double), ("lidar_ms", C.c_double), ("occupancy_ms", C.c_double),
                ("reset_ms", C.c_double), ("step_launches", C.c_int64), ("lidar_launches", C.c_int64),
                ("occupancy_launches", C.c_int64), ("reset_launches", C.c_int64),
                ("policy_ms", C.c_double), ("policy_launches", C.c_int64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class RdGapFollower(C.Structure):
    """rd_gap_follower (include/rd_env.h): the follow-the-gap controller's constants + scan geometry."""
    _fields_ = [(n, C.c_double) for n in (
        "lookahead", "vehicle_width", "minimum_gap_length", "median_dev_threshold", "kp", "ki", "kd",
        "max_vehicle_speed", "max_steering_angle", "speed_limit_angle", "scan_dt",
        "angle_min", "angle_increment", "range_max", "pct_gamma")] + [(n, C.c_int32) for n in (
        "arc_first", "arc_last", "filter_width", "pct_lo", "pct_hi", "reserved")] + [
        ("speed_scale", C.c_double), ("speed_gain", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class RdDreamerWeights(C.Structure):
    """rd_dreamer_weights (include/rd_env.h): host pointers to a Dreamer checkpoint's arrays, Keras layout."""
    _fields_ = [(n, C.c_int32) for n in ("stoch", "deter", "hidden", "embed", "actor_units", "actor_layers")] + [
        (n, C.c_void_p) for n in ("gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "obs1_w", "obs1_b",
                                  "obs2_w", "obs2_b")] + [
        ("actor_w", C.c_void_p * 8), ("actor_b", C.c_void_p * 8), ("bn", C.c_void_p),
        ("init_std", C.c_float), ("min_std", C.c_float), ("mean_scale", C.c_float), ("bn_eps", C.c_float),
        ("n_samples", C.c_int32), ("precision", C.c_int32)]


class RdDreamerExploration(C.Structure):
    """rd_dreamer_exploration: the training-mode exploration schedule and its env-step counter."""
    _fields_ = [("amount", C.c_double), ("decay", C.c_double), ("min_amount", C.c_double), ("env_steps", C.c_int64)]


class RdStoreConfig(C.Structure):
    """rd_store_config (include/rd_env.h): the device-resident episode store."""
    _fields_ = [("capacity_rows", C.c_int32), ("precision", C.c_int32), ("keep_obs", C.c_int32), ("reset_mode", C.c_int32),
                ("seed", C.c_uint64)]


class RdStoreBatch(C.Structure):
    """rd_store_batch: device pointers of a sampled [B, L, ...] batch (NULL = not produced)."""
    _fields_ = [(n, C.c_void_p) for n in (
        "lidar_dev", "occupancy_dev", "pose_dev", "velocity_dev", "speed_dev", "action_dev", "reward_dev", "discount_dev",
        "progress_dev", "time_dev", "episode_id_dev", "start_dev")]


class RdStoreSummary(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "committed", "held", "held_rows", "evicted", "invalid_requests", "draws", "capacity_rows", "max_episode_steps")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class RdStoreEpisode(C.Structure):
    _fields_ = [("id", C.c_int64), ("env", C.c_int64), ("length", C.c_int64)]


class RdStoreImportRows(C.Structure):
    """rd_store_import_rows: device pointers and element types (STORE_U8 / F16 / F32 / F64) of staged import rows."""
    KEYS = ("lidar", "occupancy", "pose", "velocity", "speed", "action", "reward", "discount", "progress", "time")
    _fields_ = [(k + "_dev", C.c_void_p) for k in KEYS] + [(k + "_type", C.c_int32) for k in KEYS]


class RdStoreImportSummary(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("imported", "held", "held_rows", "evicted", "capacity_rows")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


STORE_IMPORTED_ID0 = 1 << 62   # RD_STORE_IMPORTED_ID0
STORE_U8, STORE_F16, STORE_F32, STORE_F64 = 1, 2, 4, 8
STORE_LIDAR, STORE_POSE, STORE_VELOCITY, STORE_SPEED, STORE_OCCUPANCY = 1, 2, 4, 8, 16
STORE_KEYS = {"lidar": STORE_LIDAR, "pose": STORE_POSE, "velocity": STORE_VELOCITY, "speed": STORE_SPEED,
              "lidar_occupancy": STORE_OCCUPANCY}
STORE_POLICY_GAP_FOLLOWER, STORE_POLICY_DREAMER, STORE_POLICY_DREAMER_TRAIN = 0, 1, 2

RD_NOISE_ZERO, RD_NOISE_PHILOX, RD_NOISE_EXPLICIT = 0, 1, 2
RD_DREAMER_DEBUG_FLOATS = 68
RD_PRECISION_TF32X3, RD_PRECISION_TF32 = 0, 1

EXPORTS = (
    "rd_default_config", "rd_create", "rd_destroy", "rd_last_error", "rd_abi_version", "rd_upload_map",
    "rd_assign_maps", "rd_reset", "rd_step", "rd_lidar_cast", "rd_occupancy_obs", "rd_dynamics", "rd_reward_done",
    "rd_get_state", "rd_set_state", "rd_read_stats", "rd_launch_count", "rd_enable_timing", "rd_read_timing",
    "rd_host_init", "rd_reset_host", "rd_step_host", "rd_step_host_begin", "rd_step_host_end",
    "rd_gap_follower_defaults", "rd_policy_gap_follower_init", "rd_policy_gap_follower", "rd_rollout_gap_follower",
    "rd_policy_dreamer_init", "rd_policy_dreamer", "rd_policy_dreamer_get_state", "rd_policy_dreamer_set_state",
    "rd_rollout_dreamer", "rd_policy_dreamer_set_exploration", "rd_policy_dreamer_get_exploration",
    "rd_policy_dreamer_train", "rd_rollout_dreamer_train", "rd_policy_dreamer_set_weights",
    "rd_store_init", "rd_store_reset", "rd_store_step", "rd_rollout_store", "rd_store_sample", "rd_store_info",
    "rd_store_import_init", "rd_store_import", "rd_store_import_info",
)

LIB_PATH = Path(__file__).resolve().parent / "librd_env.so"
_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load_library() -> C.CDLL:
    """Load librd_env.so (built in-tree by __graft_entry__.build() / `make -C racing_dreamer_b200/csrc`)."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("RD_ENV_LIB") or LIB_PATH)   # RD_ENV_LIB: a prebuilt variant (tuning sweeps)
    if not path.exists():
        raise NativeLibraryError(
            f"{path} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
            "There is no CPU fallback for the env step.")
    lib = C.CDLL(str(path))
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise NativeLibraryError(f"{path} does not export {name}")
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.rd_default_config.argtypes = [C.POINTER(RdConfig)]
    lib.rd_default_config.restype = None
    lib.rd_create.argtypes = [C.POINTER(RdConfig), C.POINTER(vp)]
    lib.rd_create.restype = i32
    lib.rd_destroy.argtypes = [vp]
    lib.rd_destroy.restype = None
    lib.rd_last_error.argtypes = [vp]
    lib.rd_last_error.restype = C.c_char_p
    lib.rd_abi_version.argtypes = []
    lib.rd_abi_version.restype = i32
    lib.rd_upload_map.argtypes = [vp, i32, vp, i32, i32, i32, vp, i32, C.c_double, C.c_double, C.c_double,
                                  i32, i32, i32, vp, i32, vp, i32]
    lib.rd_upload_map.restype = i32
    lib.rd_assign_maps.argtypes = [vp, vp]
    lib.rd_assign_maps.restype = i32
    lib.rd_reset.argtypes = [vp, vp, i32, C.POINTER(RdOutputs), vp]
    lib.rd_reset.restype = i32
    lib.rd_step.argtypes = [vp, vp, C.POINTER(RdOutputs), vp]
    lib.rd_step.restype = i32
    lib.rd_host_init.argtypes = [vp, i32, C.POINTER(RdOutputs)]
    lib.rd_host_init.restype = i32
    lib.rd_reset_host.argtypes = [vp, vp, i32]
    lib.rd_reset_host.restype = i32
    lib.rd_step_host.argtypes = [vp, vp]
    lib.rd_step_host.restype = i32
    lib.rd_step_host_begin.argtypes = [vp, vp]
    lib.rd_step_host_begin.restype = i32
    lib.rd_step_host_end.argtypes = [vp]
    lib.rd_step_host_end.restype = i32
    lib.rd_lidar_cast.argtypes = [vp, vp, vp, i32, vp, vp]
    lib.rd_lidar_cast.restype = i32
    lib.rd_occupancy_obs.argtypes = [vp, vp, vp, i32, vp, vp]
    lib.rd_occupancy_obs.restype = i32
    lib.rd_dynamics.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.rd_dynamics.restype = i32
    lib.rd_reward_done.argtypes = [vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.rd_reward_done.restype = i32
    lib.rd_get_state.argtypes = [vp, vp, vp, vp]
    lib.rd_get_state.restype = i32
    lib.rd_set_state.argtypes = [vp, vp, vp, vp]
    lib.rd_set_state.restype = i32
    lib.rd_read_stats.argtypes = [vp, C.POINTER(RdStats), i32, vp]
    lib.rd_read_stats.restype = i32
    lib.rd_launch_count.argtypes = [vp]
    lib.rd_launch_count.restype = i64
    lib.rd_enable_timing.argtypes = [vp, i32]
    lib.rd_enable_timing.restype = i32
    lib.rd_read_timing.argtypes = [vp, C.POINTER(RdTiming), i32]
    lib.rd_read_timing.restype = i32
    lib.rd_gap_follower_defaults.argtypes = [C.POINTER(RdConfig), C.POINTER(RdGapFollower)]
    lib.rd_gap_follower_defaults.restype = None
    lib.rd_policy_gap_follower_init.argtypes = [vp, C.POINTER(RdGapFollower)]
    lib.rd_policy_gap_follower_init.restype = i32
    lib.rd_policy_gap_follower.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.rd_policy_gap_follower.restype = i32
    lib.rd_rollout_gap_follower.argtypes = [vp, i32, C.POINTER(RdOutputs), vp, vp]
    lib.rd_rollout_gap_follower.restype = i32
    lib.rd_policy_dreamer_init.argtypes = [vp, C.POINTER(RdDreamerWeights)]
    lib.rd_policy_dreamer_init.restype = i32
    lib.rd_policy_dreamer.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    lib.rd_policy_dreamer.restype = i32
    lib.rd_policy_dreamer_get_state.argtypes = [vp, vp, vp, vp, vp]
    lib.rd_policy_dreamer_get_state.restype = i32
    lib.rd_policy_dreamer_set_state.argtypes = [vp, vp, vp, vp, vp]
    lib.rd_policy_dreamer_set_state.restype = i32
    lib.rd_rollout_dreamer.argtypes = [vp, i32, C.POINTER(RdOutputs), vp, i32, vp]
    lib.rd_rollout_dreamer.restype = i32
    lib.rd_policy_dreamer_set_exploration.argtypes = [vp, C.POINTER(RdDreamerExploration)]
    lib.rd_policy_dreamer_set_exploration.restype = i32
    lib.rd_policy_dreamer_get_exploration.argtypes = [vp, C.POINTER(RdDreamerExploration)]
    lib.rd_policy_dreamer_get_exploration.restype = i32
    lib.rd_policy_dreamer_train.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.rd_policy_dreamer_train.restype = i32
    lib.rd_rollout_dreamer_train.argtypes = [vp, i32, C.POINTER(RdOutputs), vp, i32, vp]
    lib.rd_rollout_dreamer_train.restype = i32
    lib.rd_policy_dreamer_set_weights.argtypes = [vp, C.POINTER(RdDreamerWeights), i32, vp]
    lib.rd_policy_dreamer_set_weights.restype = i32
    lib.rd_store_init.argtypes = [vp, C.POINTER(RdStoreConfig)]
    lib.rd_store_init.restype = i32
    lib.rd_store_reset.argtypes = [vp, C.POINTER(RdOutputs), vp]
    lib.rd_store_reset.restype = i32
    lib.rd_store_step.argtypes = [vp, vp, C.POINTER(RdOutputs), vp]
    lib.rd_store_step.restype = i32
    lib.rd_rollout_store.argtypes = [vp, i32, i32, C.POINTER(RdOutputs), vp, i32, vp]
    lib.rd_rollout_store.restype = i32
    lib.rd_store_sample.argtypes = [vp, i32, i32, i32, vp, vp, C.POINTER(RdStoreBatch), vp]
    lib.rd_store_sample.restype = i32
    lib.rd_store_info.argtypes = [vp, C.POINTER(RdStoreSummary), vp, i64, vp]
    lib.rd_store_info.restype = i32
    lib.rd_store_import_init.argtypes = [vp, i32]
    lib.rd_store_import_init.restype = i32
    lib.rd_store_import.argtypes = [vp, i32, vp, C.POINTER(RdStoreImportRows), vp]
    lib.rd_store_import.restype = i32
    lib.rd_store_import_info.argtypes = [vp, C.POINTER(RdStoreImportSummary), vp, i64, vp]
    lib.rd_store_import_info.restype = i32
    if lib.rd_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f"{path}: ABI version {lib.rd_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return lib


def default_config() -> RdConfig:
    cfg = RdConfig()
    load_library().rd_default_config(C.byref(cfg))
    return cfg
