"""ctypes binding of libdekf_b200.so (include/dekf_b200.h).  Fails loudly: there is no fallback."""
import ctypes as C
import os

from .params import DekfConfig

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "libdekf_b200.so")

dp = C.POINTER(C.c_double)
up = C.POINTER(C.c_uint8)
ip = C.POINTER(C.c_int32)

# every symbol include/dekf_b200.h declares
SYMBOLS = [
    "dekf_config_default_go1", "dekf_config_default_cassie", "dekf_config_default_pogox", "dekf_create",
    "dekf_destroy", "dekf_reset", "dekf_set_stream", "dekf_get_stream", "dekf_last_error", "dekf_num_joints", "dekf_state_dim",
    "dekf_ekf_step", "dekf_mhe_step", "dekf_step", "dekf_step_host", "dekf_mhe_step_host", "dekf_ekf_step_host",
    "dekf_run", "dekf_run_host", "dekf_run_host_f32", "dekf_run_host_f32io", "dekf_synchronize", "dekf_get_arrival_cost",
    "dekf_get_arrival_cov", "dekf_get_p_vo", "dekf_get_R_sb", "dekf_get_ekf_cov", "dekf_get_window_vo_count", "dekf_get_window", "dekf_get_window_cov", "dekf_get_foot_window", "dekf_get_constrained_window", "dekf_get_window_cross_cov", "dekf_get_host", "dekf_debug_taps", "dekf_get_qp_info", "dekf_get_resweep_info", "dekf_add_state_rows",
    "dekf_launch_count", "dekf_device_bytes", "dekf_profile_enable", "dekf_profile_read", "dekf_measure_fma_peak",
    "dekf_measure_copy_bw",
]


class DekfInputs(C.Structure):
    _fields_ = [("gyro", C.c_void_p), ("accel", C.c_void_p), ("imu_time", C.c_void_p), ("joint_pos", C.c_void_p),
                ("joint_vel", C.c_void_p), ("foot_force", C.c_void_p), ("vo_flag", C.c_void_p),
                ("vo_quat", C.c_void_p), ("vo_time_pre", C.c_void_p), ("vo_time_now", C.c_void_p),
                ("vo_rel_p", C.c_void_p), ("quat", C.c_void_p)]


class DekfInputsF32(C.Structure):
    """dekf_inputs_f32: gyro / accel / joint_pos / joint_vel / foot_force point at float32 streams, the rest at float64."""
    _fields_ = [("gyro", C.c_void_p), ("accel", C.c_void_p), ("imu_time", C.c_void_p), ("joint_pos", C.c_void_p),
                ("joint_vel", C.c_void_p), ("foot_force", C.c_void_p), ("vo_flag", C.c_void_p),
                ("vo_quat", C.c_void_p), ("vo_time_pre", C.c_void_p), ("vo_time_now", C.c_void_p),
                ("vo_rel_p", C.c_void_p)]


class DekfOutputs(C.Structure):
    _fields_ = [("quat", C.c_void_p), ("x", C.c_void_p), ("v_body", C.c_void_p), ("contact", C.c_void_p),
                ("status", C.c_void_p)]


_LIB = None


def load():
    """Load the CUDA library; raises if it has not been built (run ``python -m decentralized_ekf_mhe_b200.build``)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so_path = os.environ.get("DEKF_B200_SO", SO_PATH)  # tuning variants of the library (tools/); the default is the product build
    if not os.path.exists(so_path):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -m decentralized_ekf_mhe_b200.build` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the estimator hot path.")
    L = C.CDLL(so_path)
    hp = C.c_void_p
    cfgp = C.POINTER(DekfConfig)
    for name in ("dekf_config_default_go1", "dekf_config_default_cassie", "dekf_config_default_pogox"):
        getattr(L, name).argtypes = [cfgp]
    L.dekf_create.argtypes = [cfgp, C.POINTER(hp)]
    for name in ("dekf_destroy", "dekf_reset", "dekf_synchronize"):
        getattr(L, name).argtypes = [hp]
    L.dekf_set_stream.argtypes = [hp, C.c_void_p]
    L.dekf_get_stream.argtypes = [hp]
    L.dekf_get_stream.restype = C.c_void_p
    L.dekf_last_error.argtypes = [hp]
    L.dekf_last_error.restype = C.c_char_p
    L.dekf_num_joints.argtypes = [hp]
    L.dekf_state_dim.argtypes = [hp]
    L.dekf_ekf_step.argtypes = [hp, C.POINTER(DekfInputs), C.POINTER(DekfOutputs)]
    L.dekf_ekf_step_host.argtypes = [hp, C.POINTER(DekfInputs), C.POINTER(DekfOutputs)]
    L.dekf_run_host_f32.argtypes = [hp, C.c_int32, C.c_int32, C.POINTER(DekfInputsF32), C.c_void_p, C.POINTER(DekfOutputs), C.c_int32]
    # dekf_outputs_f32 has the layout of dekf_outputs (five pointers); quat / x / v_body point at float32 arrays
    L.dekf_run_host_f32io.argtypes = [hp, C.c_int32, C.c_int32, C.POINTER(DekfInputsF32), C.c_void_p, C.POINTER(DekfOutputs), C.c_int32]
    for name in ("dekf_run", "dekf_run_host"):
        getattr(L, name).argtypes = [hp, C.c_int32, C.c_int32, C.POINTER(DekfInputs), C.c_void_p, C.POINTER(DekfOutputs),
                                     C.c_int32]
    for name in ("dekf_mhe_step", "dekf_step", "dekf_step_host", "dekf_mhe_step_host"):
        getattr(L, name).argtypes = [hp, C.c_int32, C.POINTER(DekfInputs), C.POINTER(DekfOutputs)]
    L.dekf_get_arrival_cost.argtypes = [hp, C.c_void_p, C.c_void_p]
    L.dekf_get_arrival_cov.argtypes = [hp, C.c_void_p, C.c_void_p]
    for name in ("dekf_get_p_vo", "dekf_get_R_sb", "dekf_get_ekf_cov", "dekf_get_window_vo_count"):
        getattr(L, name).argtypes = [hp, C.c_void_p]
    L.dekf_get_window.argtypes = [hp, C.c_void_p, ip]
    L.dekf_get_window_cov.argtypes = [hp, C.c_void_p, ip]
    L.dekf_get_foot_window.argtypes = [hp, C.c_void_p, C.c_void_p, ip]
    L.dekf_get_constrained_window.argtypes = [hp, C.c_void_p, C.c_void_p, C.c_void_p, ip]
    L.dekf_get_window_cross_cov.argtypes = [hp, C.c_void_p, C.c_void_p, ip]
    L.dekf_get_host.argtypes = [hp, C.c_int32, C.c_void_p]
    L.dekf_debug_taps.argtypes = [hp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.dekf_get_qp_info.argtypes = [hp, C.c_void_p, C.c_void_p]
    L.dekf_add_state_rows.argtypes = [hp, C.c_int32, dp, dp, dp]
    L.dekf_get_resweep_info.argtypes = [hp, C.c_void_p, C.c_void_p]
    L.dekf_profile_enable.argtypes = [hp, C.c_int32]
    L.dekf_profile_read.argtypes = [hp, dp, C.POINTER(C.c_int64)]
    L.dekf_measure_fma_peak.argtypes = [C.c_int32, C.c_int32, dp]
    L.dekf_measure_copy_bw.argtypes = [C.c_int32, dp]
    L.dekf_launch_count.argtypes = [hp]
    L.dekf_launch_count.restype = C.c_int64
    L.dekf_device_bytes.argtypes = [hp]
    L.dekf_device_bytes.restype = C.c_int64
    _LIB = L
    return L
