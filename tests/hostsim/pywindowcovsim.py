"""ctypes driver of the smoothed-covariance host harness (tests/hostsim/window_cov_hostsim.cpp).  NOT a product path."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def build():
    so = os.path.join(HERE, "_build", "libwindowcovsim.so")
    srcs = [os.path.join(HERE, f) for f in ("window_cov_hostsim.cpp", "hostsim.cpp")] + [
        os.path.join(ROOT, "decentralized_ekf_mhe_b200", "csrc", f)
        for f in ("estimator_core.cuh", "smallmat.cuh", "kinematics.cuh", "host_setup.hpp", "box_solve.cuh", "footstate.cuh")] + [
        os.path.join(ROOT, "include", "dekf_b200.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                               os.path.join(HERE, "window_cov_hostsim.cpp")])
    return so


def run_cov(stream, cfg):
    """Go1, est_type 0, leg_odom_type 0, no state bounds.  Returns x [S][9][n], cov [S][N][81][n]: the smoothed covariances after
    every update(T) (what dekf_get_window_cov returns; blocks K = min(T+1, N) and beyond, and all of tick 0, stay NaN) and, on
    incremental handles, filt [S][81][n]: the filtered P_T read from the checkpoint ring (NaN otherwise)."""
    lib = C.CDLL(build())
    S, _, n = stream["gyro"].shape
    cfg.n_instances = n
    dp, up = C.POINTER(C.c_double), C.POINTER(C.c_ubyte)
    keep = []

    def d(name):
        a = np.ascontiguousarray(stream[name], dtype=np.float64)
        keep.append(a)
        return a.ctypes.data_as(dp)

    flag = np.ascontiguousarray(stream["vo_flag"], dtype=np.uint8)
    res = dict(x=np.full((S, 9, n), np.nan), cov=np.full((S, int(cfg.N), 81, n), np.nan), filt=np.full((S, 81, n), np.nan))
    rc = lib.windowcovsim_run(C.byref(cfg), S, d("gyro"), d("accel"), d("imu_time"), d("joint_pos"), d("joint_vel"),
                              d("foot_force"), flag.ctypes.data_as(up), d("vo_quat"), d("vo_time_pre"), d("vo_time_now"),
                              d("vo_rel_p"), res["x"].ctypes.data_as(dp), res["cov"].ctypes.data_as(dp),
                              res["filt"].ctypes.data_as(dp))
    assert rc == 0
    return res
