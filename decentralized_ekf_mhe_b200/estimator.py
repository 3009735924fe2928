"""Host-side mirror of the reference's estimator interface, batched over instances.

Reference (C++; /root/reference/src)                          here (Python over the C ABI)
  struct robot_params   DecentralEst.hpp:18-63                 robot_params
  struct robot_store    DecentralEst.hpp:65-94                 robot_store   (every field gains a trailing instance axis)
  DecentralizedEstimation::initialize/update/reset :96-104     DecentralizedEstimation.initialize/update/reset
     public x_MHE_, v_MHE_b_, R_sb_, p_vo_accmulate_ :278-285     same attribute names (torch tensors [k, n])
  orien_ekf::timerCallback  orien_ekf.cpp:77-89                orien_ekf.timerCallback
  MHEproblem::M_p, n_p  MheSrb.hpp:86-87                       DecentralizedEstimation.mhe_qp_.M_p / .n_p
  MHEproblem::solution  MheSrb.hpp:58-112 (state blocks)       DecentralizedEstimation.mhe_qp_.x_window(), BatchedEstimator.window()
  (posterior covariance of each state block; not in the reference)  DecentralizedEstimation.mhe_qp_.P_window(), BatchedEstimator.window_cov()
  (leg_odom_type 1: the same with 9 + 3L rows per state block)    the same methods, through dekf_get_foot_window
  (state-constrained handles: the same, with the active bounds)   the same methods, through dekf_get_constrained_window;
                                                                  BatchedEstimator.window_active(), mhe_qp_.active_window()
  (lag-one cross-covariances of that window; not in the reference)  DecentralizedEstimation.mhe_qp_.P_window_cross(),
                                                                  BatchedEstimator.window_cross_cov()

torch is used for device memory and streams only; all arithmetic happens in libdekf_b200.so
(sm_100a kernels).  Nothing here falls back to PyTorch or the CPU: a missing library or device raises.
"""
import ctypes as C

import torch

from . import _lib
from .params import FP32, FP64, ROBOT_IDS, DekfConfig


class DekfError(RuntimeError):
    pass


def measure_peaks(device=0):
    """Measured roofline denominators of this device: non-tensor FMA TFLOP/s (fp64, fp32) and copy GB/s."""
    L = _lib.load()
    out = {}
    v = C.c_double()
    for name, prec in (("fp64_tflops", FP64), ("fp32_tflops", FP32)):
        rc = L.dekf_measure_fma_peak(int(device), prec, C.byref(v))
        if rc != 0:
            raise DekfError(f"dekf_measure_fma_peak failed ({rc})")
        out[name] = v.value
    rc = L.dekf_measure_copy_bw(int(device), C.byref(v))
    if rc != 0:
        raise DekfError(f"dekf_measure_copy_bw failed ({rc})")
    out["copy_gbs"] = v.value
    return out


class robot_params:
    """``struct robot_params`` + the orien_ekf parameters + batch sizes (ctypes ``dekf_config`` inside)."""

    def __init__(self, robot="go1", **over):
        self.cfg = DekfConfig()
        L = _lib.load()
        {"go1": L.dekf_config_default_go1, "cassie": L.dekf_config_default_cassie,
         "pogox": L.dekf_config_default_pogox}[robot](C.byref(self.cfg))
        self.robot = robot
        self.cfg.update(**over)

    def __getattr__(self, name):
        # reference field names carry a trailing underscore (rate_, N_, p_init_std_ ...)
        cfg = object.__getattribute__(self, "cfg")
        key = name[:-1] if name.endswith("_") else name
        if hasattr(cfg, key):
            return getattr(cfg, key)
        raise AttributeError(name)


class robot_store:
    """Batched ``struct robot_store``: the per-tick sensor snapshot of all instances (device tensors,
    float64, instance axis last).  ``vo_new_`` is a uint8 tensor [n] or None."""

    FIELDS = ("imu_time_", "accel_b_", "angular_b_", "joint_states_position_", "joint_states_velocity_",
              "foot_force_", "vo_new_", "vo_quaternion_", "vo_time_pre_", "vo_time_now_",
              "vo_p_body_pre_2_body_", "quaternion_")

    def __init__(self, **kw):
        for f in self.FIELDS:
            setattr(self, f, kw.get(f))

    @classmethod
    def from_stream(cls, stream, s, with_vo=None):
        """Snapshot ``s`` of a synth.make_stream dict (tensors already on the device)."""
        vo = bool(stream["vo_flag"][s].any()) if with_vo is None else with_vo
        return cls(imu_time_=stream["imu_time"][s], accel_b_=stream["accel"][s], angular_b_=stream["gyro"][s],
                   joint_states_position_=stream["joint_pos"][s], joint_states_velocity_=stream["joint_vel"][s],
                   foot_force_=stream["foot_force"][s],
                   vo_new_=stream["vo_flag"][s] if vo else None, vo_quaternion_=stream["vo_quat"][s],
                   vo_time_pre_=stream["vo_time_pre"][s], vo_time_now_=stream["vo_time_now"][s],
                   vo_p_body_pre_2_body_=stream["vo_rel_p"][s])


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class _Handle:
    """Owns one dekf_handle (n instances on one device)."""

    def __init__(self, params, n_instances, device=0, precision="fp64", debug_taps=False):
        if not torch.cuda.is_available():
            raise DekfError("no CUDA device: the estimator hot path has no CPU fallback")
        self.L = _lib.load()
        self.params = params
        cfg = DekfConfig.from_buffer_copy(params.cfg)
        cfg.n_instances = int(n_instances)
        cfg.device = int(device)
        cfg.precision = FP32 if precision in ("fp32", FP32) else FP64
        cfg.debug_taps = int(bool(debug_taps))
        self.cfg = cfg
        self.n = int(n_instances)
        self.device = torch.device("cuda", int(device))
        self.h = C.c_void_p()
        rc = self.L.dekf_create(C.byref(cfg), C.byref(self.h))
        if rc != 0:
            raise DekfError(f"dekf_create failed with code {rc}")
        self.nl = cfg.num_legs
        self.nq = self.L.dekf_num_joints(self.h)
        self.ds = self.L.dekf_state_dim(self.h)
        # run the library on torch's current stream of that device so tensor lifetimes stay simple
        self.stream = torch.cuda.current_stream(self.device)
        self.L.dekf_set_stream(self.h, C.c_void_p(self.stream.cuda_stream))
        f64 = dict(dtype=torch.float64, device=self.device)
        self.quat = torch.zeros(4, self.n, **f64)
        self.x = torch.full((self.ds, self.n), float("nan"), **f64)
        self.v_body = torch.full((3, self.n), float("nan"), **f64)
        self.contact = torch.zeros(self.nl, self.n, dtype=torch.uint8, device=self.device)
        self.status = torch.zeros(self.n, dtype=torch.int32, device=self.device)
        self._out = _lib.DekfOutputs(_ptr(self.quat), _ptr(self.x), _ptr(self.v_body), _ptr(self.contact),
                                     _ptr(self.status))

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.L.dekf_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc, what):
        if rc != 0:
            raise DekfError(f"{what} failed ({rc}): {self.L.dekf_last_error(self.h).decode()}")

    def inputs(self, st, quat=None):
        def chk(t, rows, name):
            if t is None:
                raise DekfError(f"robot_store.{name} is not set")
            if t.dtype != torch.float64 or t.device != self.device or not t.is_contiguous():
                raise DekfError(f"robot_store.{name} must be a contiguous float64 tensor on {self.device}")
            if t.numel() != rows * self.n:
                raise DekfError(f"robot_store.{name} has {t.numel()} elements, expected {rows}x{self.n}")
            return _ptr(t)

        vo = st.vo_new_ is not None
        if vo and (st.vo_new_.dtype != torch.uint8 or st.vo_new_.numel() != self.n):
            raise DekfError("robot_store.vo_new_ must be uint8 [n]")
        return _lib.DekfInputs(
            chk(st.angular_b_, 3, "angular_b_"), chk(st.accel_b_, 3, "accel_b_"), chk(st.imu_time_, 1, "imu_time_"),
            chk(st.joint_states_position_, self.nq, "joint_states_position_"),
            chk(st.joint_states_velocity_, self.nq, "joint_states_velocity_"),
            chk(st.foot_force_, self.nl, "foot_force_"),
            _ptr(st.vo_new_) if vo else None,
            chk(st.vo_quaternion_, 4, "vo_quaternion_") if vo and st.vo_quaternion_ is not None else None,
            chk(st.vo_time_pre_, 1, "vo_time_pre_") if vo and st.vo_time_pre_ is not None else None,
            chk(st.vo_time_now_, 1, "vo_time_now_") if vo else None,
            chk(st.vo_p_body_pre_2_body_, 3, "vo_p_body_pre_2_body_") if vo and st.vo_p_body_pre_2_body_ is not None else None,
            chk(quat, 4, "quaternion_") if quat is not None else None)


def _foot_window(h, want_x, want_P):
    """Smoothed window of a foot-state handle: ([K][ds][n], [K][ds][ds][n]) float64 on the device (dekf_get_foot_window)."""
    N, ds = int(h.cfg.N), h.ds
    x = torch.empty(N, ds, h.n, dtype=torch.float64, device=h.device) if want_x else None
    P = torch.empty(N, ds, ds, h.n, dtype=torch.float64, device=h.device) if want_P else None
    K = C.c_int32()
    h.check(h.L.dekf_get_foot_window(h.h, _ptr(x) if want_x else None, _ptr(P) if want_P else None, C.byref(K)),
            "dekf_get_foot_window")
    return (x[:K.value] if want_x else None), (P[:K.value] if want_P else None)


def _constrained(h):
    return bool(h.cfg.v_box_enable or h.cfg.x_box_mask or getattr(h, "has_rows", False))


def _box_window(h, want_x, want_P, want_act):
    """Window of a state-constrained handle: ([K][9][n], [K][9][9][n] float64, [K][n] int64 active-set words) on the device
    (dekf_get_constrained_window)."""
    N = int(h.cfg.N)
    x = torch.empty(N, 9, h.n, dtype=torch.float64, device=h.device) if want_x else None
    P = torch.empty(N, 9, 9, h.n, dtype=torch.float64, device=h.device) if want_P else None
    a = torch.empty(N, h.n, dtype=torch.int32, device=h.device) if want_act else None
    K = C.c_int32()
    h.check(h.L.dekf_get_constrained_window(h.h, _ptr(x), _ptr(P), _ptr(a), C.byref(K)), "dekf_get_constrained_window")
    k = K.value
    return (x[:k] if want_x else None), (P[:k] if want_P else None), (a[:k].to(torch.int64) & 0xFFFFFFFF if want_act else None)


def _window(h):
    """Smoothed window of the last update(T): [K][9][n] float64 on the device (dekf_get_window); foot-state handles
    (leg_odom_type 1): [K][ds][n] (dekf_get_foot_window); state-constrained handles: the window QP's optimum
    (dekf_get_constrained_window)."""
    if h.cfg.leg_odom_type == 1:
        return _foot_window(h, True, False)[0]
    if _constrained(h):
        return _box_window(h, True, False, False)[0]
    w = torch.empty(int(h.cfg.N), 9, h.n, dtype=torch.float64, device=h.device)
    K = C.c_int32()
    h.check(h.L.dekf_get_window(h.h, _ptr(w), C.byref(K)), "dekf_get_window")
    return w[:K.value]


def _window_cross_cov(h, return_cov):
    """Lag-one cross-covariances of the window of the last update(T), any est_type 0 handle: [K-1][ds][ds][n] float64 on the
    device, block j = Cov(x_{T-K+1+j}, x_{T-K+2+j}), rows over the earlier state; with return_cov also the [K][ds][ds][n]
    diagonal blocks from the same pass, as (P, C) (dekf_get_window_cross_cov)."""
    N, ds = int(h.cfg.N), h.ds
    P = torch.empty(N, ds, ds, h.n, dtype=torch.float64, device=h.device) if return_cov else None
    Cc = torch.empty(max(N - 1, 1), ds, ds, h.n, dtype=torch.float64, device=h.device)
    K = C.c_int32()
    h.check(h.L.dekf_get_window_cross_cov(h.h, _ptr(P), _ptr(Cc), C.byref(K)), "dekf_get_window_cross_cov")
    k = K.value
    return (P[:k], Cc[:k - 1]) if return_cov else Cc[:k - 1]


def _window_cov(h):
    """Smoothed covariances of the last update(T): [K][9][9][n] float64 on the device (dekf_get_window_cov); foot-state
    handles (leg_odom_type 1): [K][ds][ds][n] (dekf_get_foot_window)."""
    if h.cfg.leg_odom_type == 1:
        return _foot_window(h, False, True)[1]
    if _constrained(h):
        return _box_window(h, False, True, False)[1]
    P = torch.empty(int(h.cfg.N), 9, 9, h.n, dtype=torch.float64, device=h.device)
    K = C.c_int32()
    h.check(h.L.dekf_get_window_cov(h.h, _ptr(P), C.byref(K)), "dekf_get_window_cov")
    return P[:K.value]


class _MheQpView:
    """The public members of ``MHEproblem`` callers read: M_p, n_p (MheSrb.hpp:86-87) and the state blocks of
    ``solution`` (MheSrb.hpp:58-112)."""

    def __init__(self, owner):
        self._o = owner

    def _get(self, info):
        h = self._o._hd
        M = torch.empty(h.ds * h.ds, h.n, dtype=torch.float64, device=h.device)
        v = torch.empty(h.ds, h.n, dtype=torch.float64, device=h.device)
        fn = h.L.dekf_get_arrival_cost if info else h.L.dekf_get_arrival_cov
        h.check(fn(h.h, _ptr(M), _ptr(v)), "dekf_get_arrival")
        return M.view(h.ds, h.ds, h.n), v

    @property
    def M_p(self):
        return self._get(True)[0]

    @property
    def n_p(self):
        return self._get(True)[1]

    def arrival_cov(self):
        return self._get(False)

    def x_window(self):
        """The window QP's optimum for every state of the last update(T), T >= 1: [K][9][n], K = min(T+1, N), row j =
        stage T-K+1+j (smoothed, oldest first); row K-1 equals x_MHE_ bit for bit."""
        return _window(self._o._hd)

    def P_window(self):
        """Posterior covariance of every state of the same window: [K][9][9][n], block j = stage T-K+1+j, over (p_s, v_s,
        accel bias), exactly symmetric; block K-1 is the filtered covariance of x_T."""
        return _window_cov(self._o._hd)

    def active_window(self):
        """Active bounds of every state of the same window of a state-constrained handle: [K][n] int64, bit a = lower bound of
        row a active, bit 9 + a = upper bound (dekf_get_constrained_window)."""
        return _box_window(self._o._hd, False, False, True)[2]

    def P_window_cross(self, return_cov=False):
        """Lag-one cross-covariances of the same window: [K-1][ds][ds][n], block j = Cov(x_{T-K+1+j}, x_{T-K+2+j}), rows over
        the earlier state, not symmetric; return_cov=True returns (P_window(), C) from one pass (dekf_get_window_cross_cov)."""
        return _window_cross_cov(self._o._hd, return_cov)


class DecentralizedEstimation:
    """Batched ``DecentralizedEstimation`` (DecentralEst.hpp:96-104).

    ``initialize(sub, params)`` keeps a reference to the shared ``robot_store`` like the reference keeps
    the shared_ptr (DecentralEst.cpp:11-12) and reads the snapshot at ``update(T)`` time.  ``update`` is
    ``void`` and never raises for per-instance conditions; inspect ``status_``.
    """

    def __init__(self, n_instances, device=0, precision="fp64", debug_taps=False):
        self._n, self._device, self._precision, self._taps = n_instances, device, precision, debug_taps
        self._hd = None
        self.robot_sub_ptr_ = None
        self.params_ptr_ = None
        self.mhe_qp_ = _MheQpView(self)

    # -- reference API ---------------------------------------------------------------------------
    def initialize(self, sub, params):
        self.robot_sub_ptr_, self.params_ptr_ = sub, params
        self._hd = _Handle(params, self._n, self._device, self._precision, self._taps)
        self._step_mhe(0)

    def update(self, T):
        if self._hd is None:
            raise DekfError("update() before initialize()")
        self._step_mhe(int(T))

    def reset(self):
        if self._hd is not None:
            self._hd.check(self._hd.L.dekf_reset(self._hd.h), "dekf_reset")

    # -- results (DecentralEst.hpp:278-285) ------------------------------------------------------
    @property
    def x_MHE_(self):
        return self._hd.x

    @property
    def v_MHE_b_(self):
        return self._hd.v_body

    # KF alternative, est_type_ == 1 (DecentralEst.hpp:286-291): the step outputs are x_KF_ / v_KF_b_ then
    @property
    def x_KF_(self):
        return self._hd.x

    @property
    def v_KF_b_(self):
        return self._hd.v_body

    @property
    def C_KF_(self):
        return self.mhe_qp_.arrival_cov()[0]

    @property
    def K_KF_(self):
        """Kalman gain of the last correction, ``[9, 3 * num_legs, n]`` HOST numpy array (DecentralEst.hpp:290; needs
        ``robot_params(est_type=1, kf_export_gain=1)``): dekf_get_host(DEKF_GET_KF_GAIN)."""
        import numpy as np
        h = self._hd
        K = np.empty((9 * 3 * h.nl, h.n), dtype=np.float64)
        h.check(h.L.dekf_get_host(h.h, 8, K.ctypes.data_as(C.c_void_p)), "dekf_get_host(DEKF_GET_KF_GAIN)")
        return K.reshape(9, 3 * h.nl, h.n)

    @property
    def contact_(self):
        return self._hd.contact

    @property
    def status_(self):
        return self._hd.status

    @property
    def R_sb_(self):
        h = self._hd
        R = torch.empty(9, h.n, dtype=torch.float64, device=h.device)
        h.check(h.L.dekf_get_R_sb(h.h, _ptr(R)), "dekf_get_R_sb")
        return R.view(3, 3, h.n)

    @property
    def p_vo_accmulate_(self):
        h = self._hd
        p = torch.empty(3, h.n, dtype=torch.float64, device=h.device)
        h.check(h.L.dekf_get_p_vo(h.h, _ptr(p)), "dekf_get_p_vo")
        return p

    def debug_taps(self):
        return _debug_taps(self._hd)

    # --------------------------------------------------------------------------------------------
    def _step_mhe(self, T):
        h, st = self._hd, self.robot_sub_ptr_
        if st.quaternion_ is None:
            raise DekfError("robot_store.quaternion_ is not set (imu/filter orientation)")
        inp = h.inputs(st, quat=st.quaternion_)
        h.check(h.L.dekf_mhe_step(h.h, T, C.byref(inp), C.byref(h._out)), "dekf_mhe_step")
        if st.vo_new_ is not None:
            st.vo_new_ = None  # robot_sub_ptr_->vo_new_ = false (DecentralEst.cpp:891)


class orien_ekf:
    """Batched ``orien_ekf::orien_ekf`` (orien_ekf.hpp:21-95): ``timerCallback`` runs
    get_measurement -> gyro_nonlinear_predict -> gyro_nonlinear_correct (orien_ekf.cpp:77-89)."""

    def __init__(self, params, n_instances, device=0, precision="fp64", debug_taps=False):
        self._hd = _Handle(params, n_instances, device, precision, debug_taps)

    def timerCallback(self, store):
        h = self._hd
        inp = _ekf_inputs(h, store)
        h.check(h.L.dekf_ekf_step(h.h, C.byref(inp), C.byref(h._out)), "dekf_ekf_step")

    @property
    def quaternion_(self):
        return self._hd.quat

    @property
    def Cov_q_(self):
        h = self._hd
        P = torch.empty(16, h.n, dtype=torch.float64, device=h.device)
        h.check(h.L.dekf_get_ekf_cov(h.h, _ptr(P)), "dekf_get_ekf_cov")
        return P.view(4, 4, h.n)

    @property
    def status_(self):
        return self._hd.status


def _debug_taps(h):
    """b_meas [3*legs, n], Q_meas [legs, 6, n], vo_idx [8, n], ekf_idx [3, n] of the last step."""
    f64 = dict(dtype=torch.float64, device=h.device)
    i32 = dict(dtype=torch.int32, device=h.device)
    out = dict(b_meas=torch.empty(3 * h.nl, h.n, **f64), Q_meas=torch.empty(h.nl, 6, h.n, **f64),
               vo_idx=torch.empty(8, h.n, **i32), ekf_idx=torch.empty(3, h.n, **i32))
    h.check(h.L.dekf_debug_taps(h.h, _ptr(out["b_meas"]), _ptr(out["Q_meas"]), _ptr(out["vo_idx"]),
                                _ptr(out["ekf_idx"])), "dekf_debug_taps")
    return out


def _ekf_inputs(h, st):
    vo = st.vo_new_ is not None
    return _lib.DekfInputs(_ptr(st.angular_b_), _ptr(st.accel_b_), _ptr(st.imu_time_), None, None, None,
                           _ptr(st.vo_new_) if vo else None, _ptr(st.vo_quaternion_) if vo else None, None,
                           _ptr(st.vo_time_now_) if vo else None, None, None)


class BatchedEstimator:
    """Both estimators in lock-step (EKF tick, then MHE update on its quaternion): the benchmark path.

    ``step(T, store)`` takes device tensors and is stream-ordered (no host sync);
    ``step_host(T, host_in, host_out)`` takes pinned host tensors and includes H2D/D2H + sync.
    """

    def __init__(self, params, n_instances, device=0, precision="fp64", debug_taps=False):
        self._hd = _Handle(params, n_instances, device, precision, debug_taps)
        self.n = n_instances

    @property
    def quaternion_(self):
        return self._hd.quat

    @property
    def x_MHE_(self):
        return self._hd.x

    @property
    def v_MHE_b_(self):
        return self._hd.v_body

    @property
    def contact_(self):
        return self._hd.contact

    @property
    def status_(self):
        return self._hd.status

    @property
    def mhe_qp_(self):
        return _MheQpView(self)

    @property
    def p_vo_accmulate_(self):
        h = self._hd
        p = torch.empty(3, h.n, dtype=torch.float64, device=h.device)
        h.check(h.L.dekf_get_p_vo(h.h, _ptr(p)), "dekf_get_p_vo")
        return p

    K_KF_ = DecentralizedEstimation.K_KF_

    def window(self):
        """Smoothed window of the last update(T), T >= 1 (the state blocks of MHEproblem::solution): [K][9][n] float64 on the
        device, K = min(T+1, N), row j = stage T-K+1+j; row K-1 equals x_MHE_ bit for bit.  Stream-ordered."""
        return _window(self._hd)

    def window_cov(self):
        """Smoothed covariances of the same window: [K][9][9][n] float64 on the device, block j = stage T-K+1+j, row-major
        over (p_s, v_s, accel bias), exactly symmetric; block K-1 is the filtered covariance of x_T.  Stream-ordered."""
        return _window_cov(self._hd)

    def window_cross_cov(self, return_cov=False):
        """Lag-one cross-covariances of the same window, any est_type 0 handle: [K-1][ds][ds][n] float64 on the device, block
        j = Cov(x_{T-K+1+j}, x_{T-K+2+j}) with rows over the earlier state (not symmetric); return_cov=True returns
        (window_cov(), C) from one pass.  With the diagonal blocks they determine the window's whole joint posterior,
        Cov(x_i, x_j) = C_i P_{i+1}^-1 C_{i+1} ... P_{j-1}^-1 C_{j-1}.  Stream-ordered."""
        return _window_cross_cov(self._hd, return_cov)

    def window_active(self):
        """Active bounds of every state of the same window of a state-constrained handle (v_box_enable, x_box_mask,
        add_state_rows): [K][n] int64, bit a = lower bound of row a active, bit 9 + a = upper bound; rows are the state
        components, or the add_state_rows rows in order followed by the config's component bounds.  Stream-ordered."""
        return _box_window(self._hd, False, False, True)[2]

    def step(self, T, store):
        h = self._hd
        inp = h.inputs(store)
        h.check(h.L.dekf_step(h.h, int(T), C.byref(inp), C.byref(h._out)), "dekf_step")

    def step_host(self, T, host_in, host_out):
        """host_in: dict of CPU (pinned) tensors with the synth.make_stream keys for ONE step;
        host_out: dict with optional 'quat','x','v_body','contact','status' CPU tensors."""
        h = self._hd
        vo = host_in.get("vo_flag") is not None
        inp = _lib.DekfInputs(_ptr(host_in["gyro"]), _ptr(host_in["accel"]), _ptr(host_in["imu_time"]),
                              _ptr(host_in["joint_pos"]), _ptr(host_in["joint_vel"]), _ptr(host_in["foot_force"]),
                              _ptr(host_in["vo_flag"]) if vo else None, _ptr(host_in["vo_quat"]) if vo else None,
                              _ptr(host_in["vo_time_pre"]) if vo else None, _ptr(host_in["vo_time_now"]) if vo else None,
                              _ptr(host_in["vo_rel_p"]) if vo else None, None)
        out = _lib.DekfOutputs(_ptr(host_out.get("quat")), _ptr(host_out.get("x")), _ptr(host_out.get("v_body")),
                               _ptr(host_out.get("contact")), _ptr(host_out.get("status")))
        h.check(h.L.dekf_step_host(h.h, int(T), C.byref(inp), C.byref(out)), "dekf_step_host")

    _IN_KEYS = ("gyro", "accel", "imu_time", "joint_pos", "joint_vel", "foot_force", "vo_flag", "vo_quat", "vo_time_pre",
                "vo_time_now", "vo_rel_p")
    _OUT_KEYS = ("quat", "x", "v_body", "contact", "status")

    def _run(self, fn, name, T0, S, stream, vo_steps, out, out_per_step):
        h = self._hd
        s0 = int(stream.get("_offset", 0))
        ptrs = []
        for k in self._IN_KEYS:
            t = stream.get(k)
            if t is None:
                ptrs.append(None)
                continue
            if t.shape[0] < s0 + S or not t.is_contiguous():
                raise DekfError(f"stream[{k!r}] must be contiguous with at least {s0 + S} ticks")
            ptrs.append(_ptr(t[s0]))
        inp = _lib.DekfInputs(*ptrs, None)
        o = out or {}
        if out is not None:
            outs = _lib.DekfOutputs(*[_ptr(o.get(k)) for k in self._OUT_KEYS])
        elif name == "dekf_run":
            outs = self._hd._out
        else:
            outs = _lib.DekfOutputs(None, None, None, None, None)
        mask = None
        if vo_steps is not None:
            mask = (C.c_uint8 * S)(*[1 if v else 0 for v in vo_steps[:S]])
        h.check(fn(h.h, int(T0), int(S), C.byref(inp), mask, C.byref(outs), int(bool(out_per_step))), name)

    def run(self, T0, S, stream, vo_steps=None, out=None, out_per_step=False):
        """``S`` lock-step ticks ``T0..T0+S-1`` in one library call (dekf_run).  ``stream``: dict of DEVICE tensors
        ``[ticks, rows, n]`` with the synth.make_stream keys (tick 0 of the tensors is tick ``T0`` unless
        ``stream['_offset']`` says otherwise); ``vo_steps``: per-tick bools (any instance has VO); ``out``: dict of
        device tensors (``[S, rows, n]`` when ``out_per_step``), default: the handle's own result tensors (last tick)."""
        self._run(self._hd.L.dekf_run, "dekf_run", T0, S, stream, vo_steps, out, out_per_step)

    def run_host(self, T0, S, stream, vo_steps=None, out=None, out_per_step=False):
        """Same with pinned HOST tensors: pipelined H2D | kernels | D2H, returns when the results are in host memory."""
        self._run(self._hd.L.dekf_run_host, "dekf_run_host", T0, S, stream, vo_steps, out, out_per_step)

    F32_KEYS = ("gyro", "accel", "joint_pos", "joint_vel", "foot_force")

    def run_host_f32(self, T0, S, stream, vo_steps=None, out=None, out_per_step=False):
        """run_host for sensor streams delivered in single precision (dekf_run_host_f32): ``stream[k]`` for k in F32_KEYS are
        pinned float32 host tensors (half the PCIe bytes, widened to double on the device), everything else as in run_host."""
        import torch
        h = self._hd
        s0 = int(stream.get("_offset", 0))
        ptrs = []
        for k in self._IN_KEYS:
            t = stream.get(k)
            if t is None:
                ptrs.append(None)
                continue
            want = torch.float32 if k in self.F32_KEYS else (torch.uint8 if k == "vo_flag" else torch.float64)
            if t.dtype != want or t.shape[0] < s0 + S or not t.is_contiguous():
                raise DekfError(f"stream[{k!r}] must be contiguous {want} with at least {s0 + S} ticks")
            ptrs.append(_ptr(t[s0]))
        inp = _lib.DekfInputsF32(*ptrs)
        o = out or {}
        outs = _lib.DekfOutputs(*[_ptr(o.get(k)) for k in self._OUT_KEYS]) if out is not None else _lib.DekfOutputs(None, None, None, None, None)
        mask = None
        if vo_steps is not None:
            mask = (C.c_uint8 * S)(*[1 if v else 0 for v in vo_steps[:S]])
        f32_out = out is not None and any(o.get(k) is not None and o[k].dtype == torch.float32 for k in ("quat", "x", "v_body"))
        if f32_out:
            # dekf_run_host_f32io: results rounded to float32 once on the device, 64 instead of 128 bytes per instance-tick
            for k in ("quat", "x", "v_body"):
                if o.get(k) is not None and o[k].dtype != torch.float32:
                    raise DekfError("run_host_f32: quat / x / v_body must be all float32 or all float64")
            h.check(h.L.dekf_run_host_f32io(h.h, int(T0), int(S), C.byref(inp), mask, C.byref(outs), int(bool(out_per_step))),
                    "dekf_run_host_f32io")
            return
        h.check(h.L.dekf_run_host_f32(h.h, int(T0), int(S), C.byref(inp), mask, C.byref(outs), int(bool(out_per_step))),
                "dekf_run_host_f32")

    def reset(self):
        self._hd.check(self._hd.L.dekf_reset(self._hd.h), "dekf_reset")

    def launch_count(self):
        return int(self._hd.L.dekf_launch_count(self._hd.h))

    def window_vo_count(self):
        """[n] int32: window stages whose VO row is an equality (drives the algorithmic flop tally)."""
        h = self._hd
        c = torch.empty(h.n, dtype=torch.int32, device=h.device)
        h.check(h.L.dekf_get_window_vo_count(h.h, _ptr(c)), "dekf_get_window_vo_count")
        return c

    def add_state_rows(self, a, lb, ub):
        """General inequality rows  lb[i] <= a[i] . x_k <= ub[i]  on every window state (MHEproblem::addConstraints(name, lb, ub) with
        a dependency row on x_k, MheSrb.cpp:58-68, :217-270); `a` [count][9] over (p_s, v_s, accel bias).  Before the first step."""
        import ctypes as C
        import numpy as np
        h = self._hd
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1, 9))
        lb = np.ascontiguousarray(np.asarray(lb, dtype=np.float64).reshape(-1))
        ub = np.ascontiguousarray(np.asarray(ub, dtype=np.float64).reshape(-1))
        assert lb.size == a.shape[0] == ub.size
        dp = C.POINTER(C.c_double)
        h.check(h.L.dekf_add_state_rows(h.h, a.shape[0], a.ctypes.data_as(dp), lb.ctypes.data_as(dp), ub.ctypes.data_as(dp)),
                "dekf_add_state_rows")
        h.has_rows = True

    def qp_info(self):
        """(factorisations, active bounds) [n] int32 of the last state-constrained solve (params.v_box_enable)."""
        h = self._hd
        it = torch.empty(h.n, dtype=torch.int32, device=h.device)
        na = torch.empty(h.n, dtype=torch.int32, device=h.device)
        h.check(h.L.dekf_get_qp_info(h.h, _ptr(it), _ptr(na)), "dekf_get_qp_info")
        return it, na

    def resweep_info(self):
        """(stages re-swept, VO rows among them) [n] int32 of the last tick (incremental window solve)."""
        h = self._hd
        d = torch.empty(h.n, dtype=torch.int32, device=h.device)
        v = torch.empty(h.n, dtype=torch.int32, device=h.device)
        h.check(h.L.dekf_get_resweep_info(h.h, _ptr(d), _ptr(v)), "dekf_get_resweep_info")
        return d, v

    def profile(self, enable):
        self._hd.check(self._hd.L.dekf_profile_enable(self._hd.h, int(bool(enable))), "dekf_profile_enable")

    def profile_read(self):
        """({'ekf','assemble','solve','resweep'} -> total ms, launch counts) since the last read."""
        ms = (C.c_double * 4)()
        cnt = (C.c_int64 * 4)()
        self._hd.check(self._hd.L.dekf_profile_read(self._hd.h, ms, cnt), "dekf_profile_read")
        names = ("ekf", "assemble", "solve", "resweep")
        return {k: ms[i] for i, k in enumerate(names)}, {k: cnt[i] for i, k in enumerate(names)}

    def device_bytes(self):
        return int(self._hd.L.dekf_device_bytes(self._hd.h))

    def debug_taps(self):
        return _debug_taps(self._hd)

    def close(self):
        self._hd.close()
