"""ctypes driver of the cross-covariance host harness (tests/hostsim/window_cross_hostsim.cpp).  NOT a product path."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
INPUTS = ("gyro", "accel", "imu_time", "joint_pos", "joint_vel", "foot_force", "vo_flag", "vo_quat", "vo_time_pre",
          "vo_time_now", "vo_rel_p")


def build():
    so = os.path.join(HERE, "_build", "libwindowcrosssim.so")
    srcs = [os.path.join(HERE, f) for f in ("window_cross_hostsim.cpp", "hostsim.cpp")] + [
        os.path.join(ROOT, "decentralized_ekf_mhe_b200", "csrc", f)
        for f in ("estimator_core.cuh", "smallmat.cuh", "kinematics.cuh", "host_setup.hpp", "box_solve.cuh", "box_team.cuh",
                  "box_window.cuh", "footstate.cuh")] + [os.path.join(ROOT, "include", "dekf_b200.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                               os.path.join(HERE, "window_cross_hostsim.cpp")])
    return so


def _inputs(stream, keep):
    dp, up = C.POINTER(C.c_double), C.POINTER(C.c_ubyte)
    out = []
    for name in INPUTS:
        if name == "vo_flag":
            a = np.ascontiguousarray(stream[name], dtype=np.uint8)
            out.append(a.ctypes.data_as(up))
        else:
            a = np.ascontiguousarray(stream[name], dtype=np.float64)
            out.append(a.ctypes.data_as(dp))
        keep.append(a)
    return out


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def run_nine(stream, cfg):
    """Go1, est_type 0, leg_odom_type 0, no state bounds.  Returns x [S][9][n], cov [S][N][81][n] (what dekf_get_window_cov
    returns) and cross [S][N-1][81][n] (what dekf_get_window_cross_cov returns); blocks beyond K (K-1) and tick 0 stay NaN."""
    lib = C.CDLL(build())
    S, _, n = stream["gyro"].shape
    N = int(cfg.N)
    cfg.n_instances = n
    keep = []
    r = dict(x=np.full((S, 9, n), np.nan), cov=np.full((S, N, 81, n), np.nan), cross=np.full((S, max(N - 1, 1), 81, n), np.nan))
    rc = lib.crosssim_run_nine(C.byref(cfg), S, *_inputs(stream, keep), _p(r["x"]), _p(r["cov"]), _p(r["cross"]))
    assert rc == 0
    return r


def run_foot(stream, cfg):
    """est_type 0, leg_odom_type 1, fp64.  Returns x [S][ds][n], cov [S][N][ds][ds][n] and cross [S][N-1][ds][ds][n]."""
    lib = C.CDLL(build())
    S, _, n = stream["gyro"].shape
    ds, N = 9 + 3 * stream["foot_force"].shape[1], int(cfg.N)
    cfg.n_instances = n
    keep = []
    r = dict(x=np.full((S, ds, n), np.nan), cov=np.full((S, N, ds, ds, n), np.nan),
             cross=np.full((S, max(N - 1, 1), ds, ds, n), np.nan))
    rc = lib.crosssim_run_foot(C.byref(cfg), S, *_inputs(stream, keep), _p(r["x"]), _p(r["cov"]), _p(r["cross"]))
    assert rc == 0
    return r


def run_box(stream, cfg, quat_in=None, rows=None):
    """est_type 0, leg_odom_type 0 with state constraints (serial solve); rows = (a [count][9], lb, ub) as
    dekf_add_state_rows.  Returns x [S][9][n], cov [S][N][9][9][n], act [S][N][n] (uint32), capped [S][n] and
    cross [S][N-1][9][9][n]."""
    lib = C.CDLL(build())
    dp = C.POINTER(C.c_double)
    if rows is not None:
        ra, rl, ru = (np.ascontiguousarray(np.asarray(v, dtype=np.float64)) for v in rows)
        lib.hostsim_set_rows(int(rl.size), ra.ctypes.data_as(dp), rl.ctypes.data_as(dp), ru.ctypes.data_as(dp))
    else:
        lib.hostsim_set_rows(0, None, None, None)
    S, _, n = stream["gyro"].shape
    N = int(cfg.N)
    cfg.n_instances = n
    keep = []
    qi = np.ascontiguousarray(quat_in, dtype=np.float64) if quat_in is not None else None
    r = dict(x=np.full((S, 9, n), np.nan), cov=np.full((S, N, 9, 9, n), np.nan), act=np.zeros((S, N, n), np.uint32),
             capped=np.zeros((S, n), np.uint8), cross=np.full((S, max(N - 1, 1), 9, 9, n), np.nan))
    rc = lib.crosssim_run_box(C.byref(cfg), S, *_inputs(stream, keep), _p(qi) if qi is not None else None, _p(r["x"]),
                              _p(r["cov"]), r["act"].ctypes.data_as(C.POINTER(C.c_uint32)),
                              r["capped"].ctypes.data_as(C.POINTER(C.c_ubyte)), _p(r["cross"]))
    lib.hostsim_set_rows(0, None, None, None)
    assert rc == 0
    return r
