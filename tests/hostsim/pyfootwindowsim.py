"""ctypes driver of the foot-state window host harness (tests/hostsim/foot_window_hostsim.cpp).  NOT a product path."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def build():
    so = os.path.join(HERE, "_build", "libfootwindowsim.so")
    srcs = [os.path.join(HERE, f) for f in ("foot_window_hostsim.cpp", "hostsim.cpp")] + [
        os.path.join(ROOT, "decentralized_ekf_mhe_b200", "csrc", f)
        for f in ("estimator_core.cuh", "smallmat.cuh", "kinematics.cuh", "host_setup.hpp", "box_solve.cuh", "footstate.cuh")] + [
        os.path.join(ROOT, "include", "dekf_b200.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                               os.path.join(HERE, "foot_window_hostsim.cpp")])
    return so


def run_window(stream, cfg):
    """est_type 0, leg_odom_type 1, fp64.  Returns x [S][ds][n] (foot_solve's x_T), win [S][N][ds][n], cov [S][N][ds][ds][n]
    (the window after every update(T); rows K = min(T+1, N) and beyond, and all of tick 0, stay NaN) and info [S][ds][ds][n],
    the information matrix M_T of every update."""
    lib = C.CDLL(build())
    S, _, n = stream["gyro"].shape
    nl = stream["foot_force"].shape[1]
    ds, N = 9 + 3 * nl, int(cfg.N)
    cfg.n_instances = n
    dp, up = C.POINTER(C.c_double), C.POINTER(C.c_ubyte)
    keep = []

    def d(name):
        a = np.ascontiguousarray(stream[name], dtype=np.float64)
        keep.append(a)
        return a.ctypes.data_as(dp)

    flag = np.ascontiguousarray(stream["vo_flag"], dtype=np.uint8)
    res = dict(x=np.full((S, ds, n), np.nan), win=np.full((S, N, ds, n), np.nan), cov=np.full((S, N, ds, ds, n), np.nan),
               info=np.full((S, ds, ds, n), np.nan))
    rc = lib.footwinsim_run(C.byref(cfg), S, d("gyro"), d("accel"), d("imu_time"), d("joint_pos"), d("joint_vel"),
                            d("foot_force"), flag.ctypes.data_as(up), d("vo_quat"), d("vo_time_pre"), d("vo_time_now"),
                            d("vo_rel_p"), res["x"].ctypes.data_as(dp), res["win"].ctypes.data_as(dp), res["cov"].ctypes.data_as(dp),
                            res["info"].ctypes.data_as(dp))
    assert rc == 0
    return res
