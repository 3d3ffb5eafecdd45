"""ctypes mirror of include/cavgym.h (struct layouts, constants, prototypes).

Shared by the product loader (cavgym_b200/_native.py) and by the test-side
oracle wrapper (oracle/oracle.py), which takes the same CavScenario tables.
"""
import ctypes as C

CAV_MAX_ROADS = 4
CAV_MAX_STATICS = 8
CAV_MAX_SPAWN_BOXES = 2
CAV_MAX_SPAWN_ORIENT = 4
CAV_MAX_TYPES = 8
CAV_SMALL_M = 8
CAV_MAX_BODIES = 512
CAV_AGENT_WORDS = 5
CAV_DRAWS = 3
CAV_N_STATS = 12

CAV_F64, CAV_F32 = 0, 1
CAV_BODY_DYNAMIC, CAV_BODY_PELICAN = 0, 1
CAV_FLAG_PEDESTRIAN, CAV_FLAG_SPAWN = 1, 2
CAV_AGENT_EXTERNAL, CAV_AGENT_NOOP, CAV_AGENT_RANDOM, CAV_AGENT_RANDOM_CONSTRAINED, CAV_AGENT_PROXIMITY, CAV_AGENT_ELECTION = range(6)
CAV_COLLISIONS_NONE, CAV_COLLISIONS_EGO, CAV_COLLISIONS_ALL = range(3)
STAT_NAMES = ("episodes", "interesting", "sum_t", "sum_t2", "sum_score", "sum_score2", "env_steps", "body_steps",
              "tangent", "errors", "sum_t_interesting", "sum_t2_interesting")


class CavQuad(C.Structure):
    _fields_ = [("x", C.c_double * 4), ("y", C.c_double * 4)]


class CavBodyType(C.Structure):
    _fields_ = [(name, C.c_double) for name in (
        "length", "width", "wheelbase", "min_velocity", "max_velocity", "min_throttle", "max_throttle",
        "min_steering_angle", "max_steering_angle")]


class CavSpawn(C.Structure):
    _fields_ = [("n_boxes", C.c_int32), ("n_orientations", C.c_int32), ("boxes", CavQuad * CAV_MAX_SPAWN_BOXES),
                ("orientations", C.c_double * CAV_MAX_SPAWN_ORIENT), ("velocity", C.c_double)]


class CavBody(C.Structure):
    _fields_ = [("kind", C.c_int32), ("type_id", C.c_int32), ("flags", C.c_int32), ("spawn_id", C.c_int32),
                ("agent", C.c_int32), ("reserved", C.c_int32), ("agent_epsilon", C.c_double),
                ("agent_threshold", C.c_double), ("init_state", C.c_double * 4), ("static_box", CavQuad)]


class CavEpisodeRow(C.Structure):
    _fields_ = [("env", C.c_int64), ("episode", C.c_int32), ("timesteps", C.c_int32), ("winner", C.c_int32),
                ("liveness_sum", C.c_int32)]


CAV_SNAPSHOT_VERSION = 1


class CavSnapshotLayout(C.Structure):
    _fields_ = [("version", C.c_int32), ("dtype", C.c_int32), ("m", C.c_int32), ("reserved", C.c_int32), ("k", C.c_int64),
                ("real_rows", C.c_int64), ("i32_rows", C.c_int64), ("u8_rows", C.c_int64), ("real_offset", C.c_int64),
                ("i32_offset", C.c_int64), ("u8_offset", C.c_int64), ("total_bytes", C.c_int64), ("fingerprint", C.c_uint64)]


class CavEngineState(C.Structure):
    _fields_ = [("version", C.c_int32), ("dtype", C.c_int32), ("m", C.c_int32), ("reserved", C.c_int32), ("n", C.c_int64),
                ("shard", C.c_int64), ("t_global", C.c_int64), ("seed", C.c_uint64), ("fingerprint", C.c_uint64),
                ("tau", C.c_double), ("counters", C.c_int64 * CAV_N_STATS)]


class CavRolloutRecord(C.Structure):
    _fields_ = [("observation", C.c_void_p), ("action", C.c_void_p), ("state", C.c_void_p), ("reward", C.c_void_p),
                ("done", C.c_void_p), ("winner", C.c_void_p), ("tangent", C.c_void_p), ("timestep", C.c_void_p)]


class CavScenario(C.Structure):
    _fields_ = [("n_bodies", C.c_int32), ("n_types", C.c_int32), ("n_roads", C.c_int32), ("n_statics", C.c_int32),
                ("n_spawns", C.c_int32), ("terminate_collisions", C.c_int32), ("terminate_ego_zones", C.c_int32),
                ("terminate_ego_offroad", C.c_int32), ("max_timesteps", C.c_int64),
                ("reward_win", C.c_double), ("reward_draw", C.c_double), ("cost_step", C.c_double),
                ("viewer_width", C.c_double), ("time_resolution", C.c_double),
                ("ego_maintenance_velocity", C.c_double), ("ego_max_velocity_offset", C.c_double),
                ("centre_line", C.c_double * 4), ("roads", CavQuad * CAV_MAX_ROADS),
                ("statics", CavQuad * CAV_MAX_STATICS), ("types", CavBodyType * CAV_MAX_TYPES),
                ("spawns", C.POINTER(CavSpawn)), ("bodies", C.POINTER(CavBody))]


c_engine_p = C.c_void_p
c_stream = C.c_void_p

# name -> (restype, argtypes): every symbol include/cavgym.h declares
PROTOTYPES = {
    "cavgym_create": (C.c_int, [C.POINTER(CavScenario), C.c_int64, C.c_int, C.c_int, C.c_uint64, C.POINTER(c_engine_p)]),
    "cavgym_destroy": (C.c_int, [c_engine_p]),
    "cavgym_set_shard": (C.c_int, [c_engine_p, C.c_int64]),
    "cavgym_reset": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, c_stream]),
    "cavgym_step": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_stream]),
    "cavgym_rollout": (C.c_int, [c_engine_p, C.c_int, C.c_int, c_stream]),
    "cavgym_rollout_record": (C.c_int, [c_engine_p, C.c_int, C.c_int, C.POINTER(CavRolloutRecord), c_stream]),
    "cavgym_rollout_until": (C.c_int, [c_engine_p, C.c_int, C.c_double, C.c_uint64, C.c_void_p, C.c_void_p, c_stream]),
    "cavgym_set_agent_params": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, c_stream]),
    "cavgym_regenerate_episodes": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(CavRolloutRecord), c_stream]),
    "cavgym_replay": (C.c_int, [c_engine_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_stream]),
    "cavgym_step_host": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cavgym_step_host_f32": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cavgym_reset_host": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cavgym_info": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, c_stream]),
    "cavgym_snapshot_layout": (C.c_int, [c_engine_p, C.c_int64, C.POINTER(CavSnapshotLayout)]),
    "cavgym_save_envs": (C.c_int, [c_engine_p, C.c_void_p, C.c_int64, C.c_void_p, c_stream]),
    "cavgym_load_envs": (C.c_int, [c_engine_p, C.c_void_p, C.c_int64, C.c_void_p, c_stream]),
    "cavgym_fork_envs": (C.c_int, [c_engine_p, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "cavgym_save_engine": (C.c_int, [c_engine_p, C.POINTER(CavEngineState)]),
    "cavgym_load_engine": (C.c_int, [c_engine_p, C.POINTER(CavEngineState)]),
    "cavgym_stats": (C.c_int, [c_engine_p, C.POINTER(C.c_int64)]),
    "cavgym_set_episode_log": (C.c_int, [c_engine_p, C.c_int64]),
    "cavgym_drain_episodes": (C.c_int, [c_engine_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "cavgym_error_count": (C.c_int, [c_engine_p, C.POINTER(C.c_int64)]),
    "cavgym_launch_count": (C.c_int, [c_engine_p, C.POINTER(C.c_int64)]),
    "cavgym_state_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_liveness_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_agent_state_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_action_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_timestep_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_done_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_winner_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_error_ptr": (C.c_void_p, [c_engine_p]),
    "cavgym_set_uniform_override": (C.c_int, [c_engine_p, C.c_void_p]),
    "cavgym_set_spawn_override": (C.c_int, [c_engine_p, C.c_void_p]),
    "cavgym_set_action_logging": (C.c_int, [c_engine_p, C.c_int]),
    "cavgym_set_global_timestep": (C.c_int, [c_engine_p, C.c_int64]),
    "cavgym_set_step_path": (C.c_int, [c_engine_p, C.c_int]),
    "cavgym_set_host_path": (C.c_int, [c_engine_p, C.c_int]),
    "cavgym_set_dense_path": (C.c_int, [c_engine_p, C.c_int]),
    "cavgym_set_tangent_tolerance": (C.c_int, [c_engine_p, C.c_double]),
    "cavgym_bodies_step": (C.c_int, [C.POINTER(CavBodyType), C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_int, c_stream]),
    "cavgym_geometry_probe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, c_stream]),
    "cavgym_zones_probe": (C.c_int, [C.POINTER(CavBodyType), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, c_stream]),
    "cavgym_host_alloc": (C.c_int, [C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "cavgym_host_free": (C.c_int, [C.c_void_p]),
    "cavgym_last_error": (C.c_char_p, []),
    "cavgym_version": (C.c_char_p, []),
}


def bind(lib):
    """Attach restype/argtypes for every declared symbol; raises AttributeError if one is missing."""
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    return lib
