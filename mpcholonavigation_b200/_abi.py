"""ctypes mirror of include/mppi_b200.h (the C ABI of the MPPI hot path).

This is the Python-side binding stub a maintainer would use to drive ``libmppi_b200.so``; the struct
layouts below must match the header field for field (``tests/test_abi.py`` checks sizes and offsets
against a C program compiled from the header).

``bind(lib, prefix)`` attaches argtypes/restypes for every entry point.  The same signatures are
exported by the CPU oracle with the prefix ``oracle_`` (test infrastructure), which is why the prefix
is a parameter; the product only ever binds ``mppi_``.
"""
import ctypes as C

MPPI_OK, MPPI_E_CONFIG, MPPI_E_CUDA, MPPI_E_NCCL, MPPI_E_STATE = range(5)

MODEL_DIFF_DRIVE, MODEL_OMNI, MODEL_ACKERMANN = 0, 1, 2
MOTION_MODELS = {"DiffDrive": MODEL_DIFF_DRIVE, "Omni": MODEL_OMNI, "Ackermann": MODEL_ACKERMANN}

# critic plugin class name (critics.xml) -> mppi_critic_kind
CRITIC_KINDS = {
    "ConstraintCritic": 0,
    "CostCritic": 1,
    "GoalCritic": 2,
    "GoalAngleCritic": 3,
    "ObstaclesCritic": 4,
    "PathAlignCritic": 5,
    "PathAlignLegacyCritic": 6,
    "PathAngleCritic": 7,
    "PathFollowCritic": 8,
    "PreferForwardCritic": 9,
    "TwirlingCritic": 10,
    "VelocityDeadbandCritic": 11,
}

MAX_CRITICS = 16
MAX_FOOTPRINT = 32
MAX_TIME_STEPS = 256
MAX_PATH_POINTS = 1024
NCCL_UNIQUE_ID_BYTES = 128
IPC_HANDLE_BYTES = 64
UINT32_MAX = 0xFFFFFFFF

WANT_TRAJECTORIES, WANT_CELLS, WANT_CRITIC_COSTS = 1, 2, 4
COSTMAP_HOST, COSTMAP_DEVICE = 0, 1

f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)


class Config(C.Structure):
    _fields_ = [
        ("batch_size", C.c_int32),
        ("time_steps", C.c_int32),
        ("iteration_count", C.c_int32),
        ("model_dt", C.c_float),
        ("temperature", C.c_float),
        ("gamma", C.c_float),
        ("vx_max", C.c_float),
        ("vx_min", C.c_float),
        ("vy_max", C.c_float),
        ("wz_max", C.c_float),
        ("vx_std", C.c_float),
        ("vy_std", C.c_float),
        ("wz_std", C.c_float),
        ("motion_model", C.c_int32),
        ("ackermann_min_turning_r", C.c_float),
        ("regenerate_noises", C.c_int32),
        ("seed", C.c_uint64),
        ("device", C.c_int32),
        ("shard_offset", C.c_int64),
        ("shard_total", C.c_int64),
    ]


class CriticDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("enabled", C.c_int32),
        ("cost_power", C.c_uint32),
        ("cost_weight", C.c_float),
        ("threshold_to_consider", C.c_float),
        ("offset_from_furthest", C.c_int32),
        ("trajectory_point_step", C.c_int32),
        ("max_path_occupancy_ratio", C.c_float),
        ("use_path_orientations", C.c_int32),
        ("max_angle_to_furthest", C.c_float),
        ("forward_preference", C.c_int32),
        ("consider_footprint", C.c_int32),
        ("collision_cost", C.c_float),
        ("critical_cost", C.c_float),
        ("near_goal_distance", C.c_float),
        ("repulsion_weight", C.c_float),
        ("critical_weight", C.c_float),
        ("collision_margin_distance", C.c_float),
        ("cost_scaling_factor", C.c_float),
        ("inflation_radius", C.c_float),
        ("deadband_velocities", C.c_float * 3),
    ]


class RobotDesc(C.Structure):
    _fields_ = [
        ("footprint_size", C.c_int32),
        ("footprint_x", C.c_double * MAX_FOOTPRINT),
        ("footprint_y", C.c_double * MAX_FOOTPRINT),
        ("inscribed_radius", C.c_double),
        ("circumscribed_radius", C.c_double),
        ("inflation_layer_found", C.c_int32),
        ("inflation_cost_scaling_factor", C.c_double),
        ("track_unknown", C.c_int32),
    ]


class Costmap(C.Structure):
    _fields_ = [
        ("cells", u8p),
        ("size_x", C.c_uint32),
        ("size_y", C.c_uint32),
        ("resolution", C.c_double),
        ("origin_x", C.c_double),
        ("origin_y", C.c_double),
    ]


class CycleIn(C.Structure):
    _fields_ = [
        ("pose_x", C.c_double),
        ("pose_y", C.c_double),
        ("pose_yaw", C.c_double),
        ("speed_vx", C.c_double),
        ("speed_vy", C.c_double),
        ("speed_wz", C.c_double),
        ("goal_x", C.c_double),
        ("goal_y", C.c_double),
        ("goal_checker_xy_tolerance", C.c_double),
        ("path_size", C.c_int32),
        ("path_x", f32p),
        ("path_y", f32p),
        ("path_yaw", f32p),
        ("costmap", Costmap),
    ]


class CycleOut(C.Structure):
    _fields_ = [
        ("control_vx", f32p),
        ("control_vy", f32p),
        ("control_wz", f32p),
        ("fail_flag", C.c_int32),
        ("furthest_reached_path_point", C.c_uint32),
        ("device_ms", C.c_float),
    ]


class GroupInputs(C.Structure):
    """mppi_group_inputs: cycle inputs of a bound group in device memory, one row per member"""
    _fields_ = [
        ("state", C.c_void_p),                      # const double [n][8]
        ("goal_checker_xy_tolerance", C.c_void_p),  # const double [n]
        ("path_size", C.c_void_p),                  # const int32 [n]
        ("path", C.c_void_p),                       # const float [n][3][path_stride]
        ("path_stride", C.c_int32),
    ]


H = C.c_void_p  # opaque handle

# name -> (restype, argtypes); names are without prefix
SIGNATURES = {
    "config_default": (None, [C.POINTER(Config)]),
    "critic_default": (None, [C.c_int32, C.POINTER(CriticDesc)]),
    "create": (C.c_int, [C.POINTER(Config), C.POINTER(H)]),
    "destroy": (None, [H]),
    "reset": (C.c_int, [H]),
    "set_critics": (C.c_int, [H, C.POINTER(CriticDesc), C.c_int32]),
    "set_robot": (C.c_int, [H, C.POINTER(RobotDesc)]),
    "set_speed_limit": (C.c_int, [H, C.c_double, C.c_int32]),
    "get_constraints": (C.c_int, [H, f32p]),
    "set_noise": (C.c_int, [H, f32p, f32p, f32p]),
    "generate_noise": (C.c_int, [H, C.c_uint64]),
    "get_noise": (C.c_int, [H, f32p, f32p, f32p]),
    "set_control_sequence": (C.c_int, [H, f32p, f32p, f32p]),
    "get_control_sequence": (C.c_int, [H, f32p, f32p, f32p]),
    "shift_control_sequence": (C.c_int, [H]),
    "optimize": (C.c_int, [H, C.POINTER(CycleIn), C.POINTER(CycleOut)]),
    "eval_control": (C.c_int, [H, C.POINTER(CycleIn), C.c_int32, C.POINTER(CycleOut), f32p]),
    "set_control_history": (C.c_int, [H, f32p]),
    "get_control_history": (C.c_int, [H, f32p]),
    "get_trajectories": (C.c_int, [H, f32p, f32p, f32p]),
    "get_cells": (C.c_int, [H, i32p]),
    "get_costs": (C.c_int, [H, f32p]),
    "get_critic_costs": (C.c_int, [H, C.c_int32, f32p]),
    "get_optimized_trajectory": (C.c_int, [H, C.c_double, C.c_double, C.c_double, f32p]),
    "integrate_state_velocities": (C.c_int, [H, C.c_double, C.c_double, C.c_double, f32p, f32p, f32p, f32p, f32p, f32p]),
    "score_trajectories": (C.c_int, [H, C.POINTER(CycleIn), f32p, f32p, f32p, f32p, f32p, f32p, f32p, u32p, i32p]),
}

# entry points only the product library exports
PRODUCT_ONLY = {
    "last_error": (C.c_char_p, [H]),
    "abi_version": (C.c_int32, []),
    "optimize_batch": (C.c_int, [C.POINTER(H), C.POINTER(CycleIn), C.POINTER(CycleOut), C.c_int32]),
    "optimize_sharded": (C.c_int, [C.POINTER(H), C.c_int32, C.POINTER(CycleIn), C.POINTER(CycleOut)]),
    "optimize_batch_resident": (C.c_int, [C.POINTER(H), C.POINTER(CycleOut), C.c_int32]),
    "batch_bind": (C.c_int, [C.POINTER(H), C.c_int32]),
    "batch_unbind": (C.c_int, [H]),
    "batch_span_ms": (C.c_int, [C.POINTER(H), C.c_int32, f32p]),
    "optimize_group_device": (C.c_int, [C.POINTER(H), C.c_int32, C.POINTER(GroupInputs), C.POINTER(Costmap), C.POINTER(CycleOut)]),
    "debug_get_record": (C.c_int, [H, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "upload_cycle": (C.c_int, [H, C.POINTER(CycleIn)]),
    "optimize_resident": (C.c_int, [H, C.POINTER(CycleOut)]),
    "set_outputs": (C.c_int, [H, C.c_uint32]),
    "set_visualization": (C.c_int, [H, C.c_int32, C.c_int32]),
    "get_visualization": (C.c_int, [H, f32p, f32p]),
    "set_profiling": (C.c_int, [H, C.c_int32]),
    "set_timing": (C.c_int, [H, C.c_int32]),
    "set_costmap_residency": (C.c_int, [H, C.c_int32]),
    "register_costmap_memory": (C.c_int, [H, C.c_void_p, C.c_uint64]),
    "unregister_costmap_memory": (C.c_int, [H, C.c_void_p]),
    "get_profile": (C.c_int, [H, f32p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "comm_get_unique_id": (C.c_int, [u8p]),
    "comm_init": (C.c_int, [H, u8p, C.c_int32, C.c_int32]),
    "comm_get_mailbox_handle": (C.c_int, [H, u8p]),
    "comm_connect_peers": (C.c_int, [H, u8p, C.c_int32, C.c_int32]),
    "comm_destroy": (C.c_int, [H]),
}


def bind(lib, prefix, extra=None):
    """Attach signatures to ``lib`` and return {short name: function}."""
    table = dict(SIGNATURES)
    if extra:
        table.update(extra)
    out = {}
    for name, (res, args) in table.items():
        fn = getattr(lib, prefix + name)
        fn.restype = res
        fn.argtypes = args
        out[name] = fn
    return out
