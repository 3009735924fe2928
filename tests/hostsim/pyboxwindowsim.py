"""ctypes driver of the constrained-window host harness (tests/hostsim/box_window_hostsim.cpp).  NOT a product path."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def build():
    so = os.path.join(HERE, "_build", "libboxwindowsim.so")
    srcs = [os.path.join(HERE, f) for f in ("box_window_hostsim.cpp", "hostsim.cpp")] + [
        os.path.join(ROOT, "decentralized_ekf_mhe_b200", "csrc", f)
        for f in ("estimator_core.cuh", "smallmat.cuh", "kinematics.cuh", "host_setup.hpp", "box_solve.cuh", "box_team.cuh",
                  "box_window.cuh", "footstate.cuh")] + [os.path.join(ROOT, "include", "dekf_b200.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                               os.path.join(HERE, "box_window_hostsim.cpp")])
    return so


def run_window(stream, cfg, quat_in=None, rows=None):
    """est_type 0, leg_odom_type 0 with state constraints; rows = (a [count][9], lb, ub) as dekf_add_state_rows.  Returns x
    [S][9][n] (the step's x_T), status [S][n], win [S][N][9][n], cov [S][N][9][9][n], act [S][N][n] (uint32) and capped [S][n]
    (the window after every update(T); rows K = min(T+1, N) and beyond, and all of tick 0, stay NaN / 0)."""
    lib = C.CDLL(build())
    dp, up, ip = C.POINTER(C.c_double), C.POINTER(C.c_ubyte), C.POINTER(C.c_int32)
    if rows is not None:
        ra, rl, ru = (np.ascontiguousarray(np.asarray(v, dtype=np.float64)) for v in rows)
        lib.hostsim_set_rows(int(rl.size), ra.ctypes.data_as(dp), rl.ctypes.data_as(dp), ru.ctypes.data_as(dp))
    else:
        lib.hostsim_set_rows(0, None, None, None)
    S, _, n = stream["gyro"].shape
    N = int(cfg.N)
    cfg.n_instances = n
    keep = []

    def d(name):
        a = np.ascontiguousarray(stream[name], dtype=np.float64)
        keep.append(a)
        return a.ctypes.data_as(dp)

    flag = np.ascontiguousarray(stream["vo_flag"], dtype=np.uint8)
    qi = np.ascontiguousarray(quat_in, dtype=np.float64) if quat_in is not None else None
    res = dict(x=np.full((S, 9, n), np.nan), status=np.zeros((S, n), np.int32), win=np.full((S, N, 9, n), np.nan),
               cov=np.full((S, N, 9, 9, n), np.nan), act=np.zeros((S, N, n), np.uint32), capped=np.zeros((S, n), np.uint8))
    rc = lib.boxwinsim_run(C.byref(cfg), S, d("gyro"), d("accel"), d("imu_time"), d("joint_pos"), d("joint_vel"),
                           d("foot_force"), flag.ctypes.data_as(up), d("vo_quat"), d("vo_time_pre"), d("vo_time_now"),
                           d("vo_rel_p"), qi.ctypes.data_as(dp) if qi is not None else None,
                           res["x"].ctypes.data_as(dp), res["status"].ctypes.data_as(ip), res["win"].ctypes.data_as(dp),
                           res["cov"].ctypes.data_as(dp), res["act"].ctypes.data_as(C.POINTER(C.c_uint32)),
                           res["capped"].ctypes.data_as(up))
    lib.hostsim_set_rows(0, None, None, None)
    assert rc == 0
    return res
