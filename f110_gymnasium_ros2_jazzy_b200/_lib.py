"""ctypes binding of libf110_b200.so (the C ABI in include/f110_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is visible the
import / first use raises, loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("F110_B200_LIB") or os.path.join(_HERE, "csrc", "libf110_b200.so")   # env override: tuning builds only

F110_ABI_VERSION = 2
F110_NUM_PARAMS = 18
F110_NUM_STATS = 8
F110_MAX_AGENTS = 16
F110_FLAG_COUNT_LOOKUPS = 1
F110_FLAG_NARROW_FRACTION = 2
F110_HOST_MERGE_ADJACENT = 1
F110_MAX_MAPS = 256

F110_OK = 0
F110_ERR_INVALID, F110_ERR_MAP_NOT_SET, F110_ERR_CUDA, F110_ERR_INDEX = -1, -2, -3, -4
F110_ERR_POSE_COUNT, F110_ERR_INTEGRATOR, F110_ERR_NO_DEVICE = -5, -6, -7

# every symbol include/f110_b200.h declares
EXPORTS = ["f110_last_error", "f110_abi_version", "f110_create", "f110_destroy", "f110_set_map", "f110_set_map_image", "f110_get_map", "f110_set_maps",
           "f110_map_count", "f110_get_map_slot", "f110_set_env_maps", "f110_set_env_maps_host", "f110_get_env_maps", "f110_set_tables",
           "f110_set_beam_tables", "f110_set_params", "f110_sim_reset", "f110_sim_reset_host", "f110_step", "f110_step_host", "f110_step_host_async", "f110_host_sync", "f110_step_host_multi",
           "f110_state_nbytes", "f110_get_state", "f110_set_state", "f110_get_stats", "f110_get_lookup_count",
           "f110_kernel_launches", "f110_max_lookups", "f110_redone_rays", "f110_get_lidar_variant", "f110_map_generation", "f110_debug_unit_timeline", "f110_set_kernel_timing", "f110_get_kernel_timing", "f110_gap_follow", "f110_gather_probe", "f110_trig_probe", "f110_hypot_probe", "f110_edt_kernel_ms", "f110_reward_create", "f110_reward_destroy",
           "f110_reward_compute", "f110_reward_create_set", "f110_reward_count", "f110_reward_compute_slots"]


class F110Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("num_envs", C.c_int32), ("num_agents", C.c_int32),
                ("num_beams", C.c_int32), ("theta_dis", C.c_int32), ("integrator", C.c_int32), ("ego_idx", C.c_int32),
                ("flags", C.c_uint32), ("host_stream_rank", C.c_uint32),
                ("fov", C.c_double), ("eps", C.c_double), ("max_range", C.c_double), ("timestep", C.c_double),
                ("lidar_dist", C.c_double), ("ttc_thresh", C.c_double), ("lidar_max", C.c_double),
                ("noise_std", C.c_double), ("seed", C.c_uint64)]


class F110StepIO(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("actions_f64", C.c_int32), ("host_flags", C.c_int32),
                ("noise", C.c_void_p), ("reset_mask", C.c_void_p), ("reset_poses", C.c_void_p),
                ("active_mask", C.c_void_p),
                ("obs", C.c_void_p), ("reward", C.c_void_p), ("terminated", C.c_void_p), ("scans_f64", C.c_void_p),
                ("scans_f32", C.c_void_p), ("state", C.c_void_p), ("collisions", C.c_void_p), ("toggles", C.c_void_p),
                ("lap_times", C.c_void_p), ("lap_counts", C.c_void_p), ("time", C.c_void_p), ("agent_poses", C.c_void_p)]


class F110MapDesc(C.Structure):
    _fields_ = [("dt", C.c_void_p), ("free_mask", C.c_void_p), ("height", C.c_int32), ("width", C.c_int32),
                ("resolution", C.c_double), ("orig_x", C.c_double), ("orig_y", C.c_double), ("orig_cos", C.c_double),
                ("orig_sin", C.c_double)]


class F110RewardConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("num_envs", "num_points", "num_beams", "device", "closed", "grace_steps_wall",
                                         "grace_steps_opp", "reserved")] + \
               [(n, C.c_double) for n in ("dt", "w_prog", "forward_sign", "alive_bonus", "w_rel_lead", "lead_clip", "w_lat",
                                          "lat_cap", "default_half_width", "lidar_max", "near_wall_dist", "w_wall",
                                          "wall_quantile", "opp_safe_dist", "w_opp", "ego_crash_penalty", "opp_crash_bonus")]


class F110Centerline(C.Structure):
    _fields_ = [("xy", C.c_void_p), ("wR", C.c_void_p), ("wL", C.c_void_p), ("num_points", C.c_int32), ("closed", C.c_int32)]


_lib = None


def load():
    """Load libf110_b200.so; raises RuntimeError if it has not been built (python __graft_entry__.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libf110_b200.so not found at %s -- build it with `python __graft_entry__.py` (or "
                           "`make -C f110_gymnasium_ros2_jazzy_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.f110_last_error.restype = C.c_char_p
    L.f110_abi_version.restype = C.c_int
    L.f110_create.argtypes = [C.POINTER(F110Config), vp, C.POINTER(vp)]
    L.f110_destroy.argtypes = [vp]
    L.f110_destroy.restype = None
    L.f110_set_map.argtypes = [vp, vp, C.c_int32, C.c_int32] + [C.c_double] * 5
    L.f110_set_map_image.argtypes = [vp, vp, C.c_int32, C.c_int32] + [C.c_double] * 5
    L.f110_get_map.argtypes = [vp, vp, C.c_int64]
    L.f110_set_maps.argtypes = [vp, C.POINTER(F110MapDesc), C.c_int32]
    L.f110_map_count.argtypes = [vp]
    L.f110_map_count.restype = C.c_int32
    L.f110_get_map_slot.argtypes = [vp, C.c_int32, vp, C.c_int64]
    L.f110_set_env_maps.argtypes = [vp, vp, vp, vp]
    L.f110_set_env_maps_host.argtypes = [vp, vp, vp]
    L.f110_get_env_maps.argtypes = [vp, vp, vp]
    L.f110_set_tables.argtypes = [vp, vp, vp]
    L.f110_set_beam_tables.argtypes = [vp, vp, vp, vp]
    L.f110_set_params.argtypes = [vp, vp, C.c_int32]
    L.f110_sim_reset.argtypes = [vp, vp, C.c_int32, vp, vp]
    L.f110_sim_reset_host.argtypes = [vp, vp, C.c_int32, vp]
    L.f110_step.argtypes = [vp, C.POINTER(F110StepIO), vp]
    L.f110_step_host.argtypes = [vp, C.POINTER(F110StepIO)]
    L.f110_step_host_async.argtypes = [vp, C.POINTER(F110StepIO)]
    L.f110_host_sync.argtypes = [vp]
    L.f110_step_host_multi.argtypes = [C.POINTER(vp), C.POINTER(F110StepIO), C.c_int32]
    L.f110_state_nbytes.argtypes = [vp]
    L.f110_state_nbytes.restype = C.c_int64
    L.f110_get_state.argtypes = [vp, vp, vp]
    L.f110_set_state.argtypes = [vp, vp, vp]
    L.f110_get_stats.argtypes = [vp, vp, C.c_int32, vp]
    L.f110_get_lookup_count.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.f110_set_kernel_timing.argtypes = [vp, C.c_int32]
    L.f110_get_kernel_timing.argtypes = [vp, vp, C.POINTER(C.c_int64)]
    L.f110_gap_follow.argtypes = [vp, C.c_int64, C.c_int64, C.c_int32, vp, C.c_int64, C.c_double, C.c_double, C.c_float,
                                  C.c_int32, C.c_int32, C.c_float, vp]
    L.f110_edt_kernel_ms.argtypes = [vp]
    L.f110_edt_kernel_ms.restype = C.c_float
    L.f110_gather_probe.argtypes = [vp, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int32, vp, C.POINTER(C.c_float), vp]
    L.f110_trig_probe.argtypes = [vp, C.c_int64, vp, vp]
    L.f110_hypot_probe.argtypes = [vp, vp, C.c_int64, vp, vp]
    L.f110_reward_create.argtypes = [C.POINTER(F110RewardConfig), vp, vp, vp, C.POINTER(vp)]
    L.f110_reward_destroy.argtypes = [vp]
    L.f110_reward_destroy.restype = None
    L.f110_reward_compute.argtypes = [vp, vp, vp, vp, vp, vp]
    L.f110_reward_create_set.argtypes = [C.POINTER(F110RewardConfig), C.POINTER(F110Centerline), C.c_int32, C.POINTER(vp)]
    L.f110_reward_count.argtypes = [vp]
    L.f110_reward_count.restype = C.c_int32
    L.f110_reward_compute_slots.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.f110_max_lookups.argtypes = [vp]
    L.f110_max_lookups.restype = C.c_int64
    L.f110_redone_rays.argtypes = [vp]
    L.f110_redone_rays.restype = C.c_int64
    L.f110_get_lidar_variant.argtypes = [vp, vp]
    L.f110_debug_unit_timeline.argtypes = [vp, vp, C.c_int64]
    L.f110_debug_unit_timeline.restype = C.c_int64
    L.f110_map_generation.argtypes = [vp]
    L.f110_map_generation.restype = C.c_int64
    L.f110_kernel_launches.argtypes = [vp]
    L.f110_kernel_launches.restype = C.c_int64
    if L.f110_abi_version() != F110_ABI_VERSION:
        raise RuntimeError("libf110_b200.so ABI %d != binding ABI %d; rebuild" % (L.f110_abi_version(), F110_ABI_VERSION))
    _lib = L
    return L


def check(rc):
    """Map C status codes onto the exceptions the reference raises for the same conditions."""
    if rc == F110_OK:
        return
    msg = load().f110_last_error().decode("utf-8", "replace")
    if rc == F110_ERR_MAP_NOT_SET:
        raise ValueError(msg)                      # laser_models.py:445-446
    if rc == F110_ERR_POSE_COUNT:
        raise ValueError(msg)                      # base_classes.py:638-639
    if rc == F110_ERR_INDEX:
        raise IndexError(msg)                      # base_classes.py:547
    if rc == F110_ERR_INTEGRATOR:
        raise SyntaxError(msg)                     # base_classes.py:399
    if rc == F110_ERR_INVALID:
        raise ValueError(msg)
    raise RuntimeError("libf110_b200: %s (code %d)" % (msg, rc))
