"""ctypes loader for libmrsb.so (the C ABI declared in include/mrsb.h).

There is no Python or CPU fallback: if the library is missing this module raises, and
mrsb_create itself fails without a CUDA device.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MRSB_LIB_PATH") or os.path.join(HERE, "libmrsb.so")  # MRSB_LIB_PATH: kernel-variant experiments only
MAX_MOTORS = 8

i32p = C.POINTER(C.c_int32)
f64p = C.POINTER(C.c_double)


class ModelParams(C.Structure):
    """mrsb_model_params == MultirotorModel::ModelParams (multirotor_model.hpp:24-88)."""
    _fields_ = [("n_motors", C.c_int32), ("ground_enabled", C.c_int32), ("takeoff_patch_enabled", C.c_int32), ("reserved_", C.c_int32),
                ("g", C.c_double), ("mass", C.c_double), ("kf", C.c_double), ("km", C.c_double), ("prop_radius", C.c_double),
                ("arm_length", C.c_double), ("body_height", C.c_double), ("motor_time_constant", C.c_double), ("max_rpm", C.c_double),
                ("min_rpm", C.c_double), ("air_resistance_coeff", C.c_double), ("ground_z", C.c_double), ("J", C.c_double * 9),
                ("allocation_matrix", C.c_double * (4 * MAX_MOTORS))]


class ControllerParams(C.Structure):
    _fields_ = [("mixer_desaturation", C.c_int32), ("reserved_", C.c_int32),
                ("rate_kp", C.c_double), ("rate_kd", C.c_double), ("rate_ki", C.c_double),
                ("att_kp", C.c_double), ("att_kd", C.c_double), ("att_ki", C.c_double), ("att_max_rate_roll_pitch", C.c_double),
                ("att_max_rate_yaw", C.c_double),
                ("vel_kp", C.c_double), ("vel_kd", C.c_double), ("vel_ki", C.c_double), ("vel_max_acceleration", C.c_double),
                ("pos_kp", C.c_double), ("pos_kd", C.c_double), ("pos_ki", C.c_double), ("pos_max_velocity", C.c_double)]


class CreateInfo(C.Structure):
    _fields_ = [("device", C.c_int32), ("n_types", C.c_int32), ("types", C.POINTER(ModelParams)), ("n_local", C.c_int64),
                ("n_global", C.c_int64), ("shard_begin", C.c_int64), ("type_of_uav", C.c_void_p), ("spawn_xyz", C.c_void_p),
                ("spawn_heading", C.c_void_p)]


class DeviceView(C.Structure):
    _fields_ = [("tile", C.c_int32), ("state_rows", C.c_int32), ("state", C.c_void_p), ("motor_rpm", C.c_void_p), ("imu_acc", C.c_void_p),
                ("ext_force", C.c_void_p), ("flags", C.c_void_p), ("input_mode", C.c_void_p), ("slot_of_uav", C.c_void_p)]


# every symbol include/mrsb.h declares: name -> (restype, argtypes)
H = C.c_void_p
_N_IDX = [H, C.c_int64, C.c_void_p]
SIGNATURES = {
    "mrsb_last_error": (C.c_char_p, []),
    "mrsb_version": (C.c_int, []),
    "mrsb_model_params_default": (None, [C.POINTER(ModelParams)]),
    "mrsb_model_params_finalize": (None, [C.POINTER(ModelParams)]),
    "mrsb_controller_params_default": (None, [C.POINTER(ControllerParams)]),
    "mrsb_mixer_allocation_of": (None, [C.POINTER(ModelParams), C.c_void_p]),
    "mrsb_bucket_layout": (C.c_int, [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]),
    "mrsb_create": (C.c_int, [C.POINTER(CreateInfo), C.POINTER(H)]),
    "mrsb_destroy": (C.c_int, [H]),
    "mrsb_sync": (C.c_int, [H]),
    "mrsb_n_local": (C.c_int64, [H]),
    "mrsb_n_global": (C.c_int64, [H]),
    "mrsb_get_stream": (C.c_void_p, [H]),
    "mrsb_set_input_actuators": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_control_group": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_attitude_rate": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_attitude": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_tilt_hdg_rate": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_acceleration_hdg_rate": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_acceleration_hdg": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_velocity_hdg_rate": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_velocity_hdg": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_input_position": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_clear_input": (C.c_int, _N_IDX),
    "mrsb_set_input": (C.c_int, [H, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32]),
    "mrsb_set_input_device": (C.c_int, [H, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32]),
    "mrsb_set_input_async": (C.c_int, [H, C.c_int32, C.c_void_p, C.c_int32]),
    "mrsb_get_positions_async": (C.c_int, [H, C.c_void_p]),
    "mrsb_set_input_rows_async": (C.c_int, [H, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "mrsb_get_observations_async": (C.c_int, [H, C.c_void_p]),
    "mrsb_set_position_subset": (C.c_int, [H, C.c_int64, C.c_void_p]),
    "mrsb_wait_uploads": (C.c_int, [H]),
    "mrsb_wait_downloads": (C.c_int, [H]),
    "mrsb_set_feedforward_acceleration_hdg_rate": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_feedforward_acceleration_hdg": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_feedforward_velocity_hdg": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_feedforward_velocity_hdg_rate": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_tracker_cmd": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_clear_feedforward": (C.c_int, _N_IDX),
    "mrsb_make_step": (C.c_int, [H, C.c_double, C.c_int32]),
    "mrsb_run": (C.c_int, [H, C.c_double, C.c_int32, C.c_int32, C.c_int32]),
    "mrsb_set_iterate_without_input": (C.c_int, [H, C.c_int32]),
    "mrsb_set_outputs": (C.c_int, [H, C.c_uint32]),
    "mrsb_get_state": (C.c_int, _N_IDX + [C.c_void_p] * 5),
    "mrsb_get_v_prev": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_get_imu_acceleration": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_state": (C.c_int, _N_IDX + [C.c_void_p] * 5),
    "mrsb_set_state_pos": (C.c_int, _N_IDX + [C.c_void_p, C.c_void_p]),
    "mrsb_respawn": (C.c_int, _N_IDX + [C.c_void_p, C.c_void_p]),
    "mrsb_respawn_masked_device": (C.c_int, [H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mrsb_snapshot_create": (C.c_int, [H, C.POINTER(C.c_int32)]),
    "mrsb_snapshot_free": (C.c_int, [H, C.c_int32]),
    "mrsb_snapshot_save": (C.c_int, [H, C.c_int32]),
    "mrsb_snapshot_restore": (C.c_int, [H, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "mrsb_snapshot_restore_device": (C.c_int, [H, C.c_int32, C.c_void_p]),
    "mrsb_snapshot_image_size": (C.c_int, [H, C.POINTER(C.c_size_t)]),
    "mrsb_snapshot_download": (C.c_int, [H, C.c_int32, C.c_void_p, C.c_size_t]),
    "mrsb_snapshot_upload": (C.c_int, [H, C.c_int32, C.c_void_p, C.c_size_t]),
    "mrsb_get_input_mode": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_crash": (C.c_int, _N_IDX),
    "mrsb_has_crashed": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_apply_force": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_get_external_force": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_external_moment": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_get_params": (C.c_int, [H, C.c_int64, C.POINTER(ModelParams)]),
    "mrsb_set_params": (C.c_int, _N_IDX + [C.POINTER(ModelParams)]),
    "mrsb_set_mixer_params": (C.c_int, _N_IDX + [C.c_int32]),
    "mrsb_set_rate_controller_params": (C.c_int, _N_IDX + [C.c_double] * 3),
    "mrsb_set_attitude_controller_params": (C.c_int, _N_IDX + [C.c_double] * 5),
    "mrsb_set_velocity_controller_params": (C.c_int, _N_IDX + [C.c_double] * 4),
    "mrsb_set_position_controller_params": (C.c_int, _N_IDX + [C.c_double] * 4),
    "mrsb_get_controller_params": (C.c_int, [H, C.c_int64, C.POINTER(ControllerParams)]),
    "mrsb_get_mixer_allocation": (C.c_int, [H, C.c_int64, C.c_void_p]),
    "mrsb_timeout_input": (C.c_int, _N_IDX),
    "mrsb_get_odometry": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_get_imu": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_get_rangefinder": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_pack_observations_device": (C.c_int, [H, C.c_void_p, C.c_int32]),
    "mrsb_set_mass": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_set_ground_z": (C.c_int, _N_IDX + [C.c_void_p]),
    "mrsb_pack_neighbours_device": (C.c_int, [H, C.c_double, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "mrsb_set_collisions": (C.c_int, [H, C.c_int32, C.c_int32, C.c_double]),
    "mrsb_handle_collisions": (C.c_int, [H]),
    "mrsb_get_collision_pairs": (C.c_int, [H, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "mrsb_set_pair_capacity": (C.c_int, [H, C.c_int64]),
    "mrsb_get_counters": (C.c_int, [H, C.c_void_p]),
    "mrsb_get_step_info": (C.c_int, [H, C.c_void_p]),
    "mrsb_get_sweep_launches": (C.c_int, [H, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "mrsb_get_timeline": (C.c_int, [H, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "mrsb_get_collision_info": (C.c_int, [H, C.c_void_p]),
    "mrsb_forces_written": (C.c_int, [H]),
    "mrsb_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "mrsb_comm_init_nccl": (C.c_int, [H, C.c_int32, C.c_int32, C.c_void_p]),
    "mrsb_exchange_mode": (C.c_int, [H]),
    "mrsb_gather_buffer": (C.c_int, [H, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "mrsb_publish_positions": (C.c_int, [H]),
    "mrsb_handle_collisions_gathered": (C.c_int, [H]),
    "mrsb_get_device_view": (C.c_int, [H, C.POINTER(DeviceView)]),
    "mrsb_microbench_fp64": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "mrsb_microbench_copy": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
}

_lib = None


def lib():
    """Load libmrsb.so; raise (never fall back) if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(or make -C mrs_multirotor_simulator_b200/csrc); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class MrsbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libmrsb error {code}: {msg}")
        self.code = code


def check(rc):
    if rc != 0:
        raise MrsbError(rc, lib().mrsb_last_error().decode(errors="replace"))
