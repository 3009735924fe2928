"""Lag-one cross-covariances of the MHE window (dekf_get_window_cross_cov): for every pair of adjacent window states the block
Cov(x_k, x_{k+1}) of the window QP's posterior, for every est_type 0 handle kind, from the backward covariance pass of that
kind with the cross block switched on (csrc/estimator_core.cuh window_cov_stage, csrc/footstate.cuh fw_cross_col,
csrc/box_window.cuh bw_cross_col).

Oracle: the oracle's window QP of the same tick (Mhe.export_qp()), its KKT matrix with the equality rows (and, for
constrained handles, a row per bound the getter reports active), solved for the unit columns of the state variables; block
(k, k+1) of that solution is the reference for C_k.  Errors are correlation-scaled, |dC_ab| / sqrt(P_k,aa P_k+1,bb) with the
oracle's diagonal.  CPU: the header code in the host build (tests/hostsim/*_hostsim.cpp).  GPU (-m gpu): the device getter
against the oracle and the host build, P of the new call against the covariance getters, invariants at size, output
invariance, the error paths and the mirrors."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "hostsim"))
GOLDEN = os.path.join(HERE, "golden", "go1_refnodes_golden.npz")
TOL64, TOL32 = 1e-8, 1e-4
# the ticks of the 9-state covariance test: T < N, T >= N without VO equalities, and T >= N with them
TICKS9 = {"ragged_n20": (1, 6, 15, 19, 25, 33, 44, 52, 61, 79), "mhe_n5": (1, 3, 4, 9, 30, 57, 80, 119),
          "mhe_n5_late": (1, 3, 4, 12, 40, 63, 79)}
# the exact foot case of the foot-window test: N = 400 without VO never marginalises
FOOT_S, FOOT_TICKS, FOOT_N = 46, (12, 20, 33, 45), 20
# the constrained-window test's handles and ticks
POGOX = dict(robot=2, num_legs=1, contact_effort_threshold=100.0, p_ib=(0.0, 0.0, 0.0), p_imu_2_opti=(0.0, 0.0, 0.0))
BOX_LO, BOX_HI = (-0.45, -0.03, -0.015), (0.55, 0.03, 0.015)
MASK = (1 << 3) | (1 << 2) | (7 << 6)
LO9 = (0, 0, -2e-4, 0.47, 0, 0, -0.004, -0.004, -0.004)
HI9 = (0, 0, 2e-4, 0.52, 0, 0, 0.004, 0.004, 0.004)
BOX_TICKS = (1, 4, 12, 19, 20, 21, 33, 47)
EINVAL, ESTATE = -1, -5   # include/dekf_b200.h


def _rows3():
    A = np.zeros((3, 9))
    A[0, 3], A[0, 5] = 1.0, 0.5
    A[1, 6], A[1, 7] = 1.0, -1.0
    A[2, 2], A[2, 8] = 1.0, 0.02
    return A, np.array([0.47, -0.003, -2e-4]), np.array([0.52, 0.003, 2e-4])


def _kind(name):
    """(config overrides, oracle overrides, rows for dekf_add_state_rows, bounded rows R [m][9]) of a constrained handle kind,
    rows in the public order of the active words."""
    if name == "vbox":
        kw = dict(v_box_enable=1, v_box_lo=BOX_LO, v_box_hi=BOX_HI)
        return kw, kw, None, np.eye(9)
    if name == "xbox":
        kw = dict(x_box_mask=MASK, x_box_lo=LO9, x_box_hi=HI9)
        return kw, kw, None, np.eye(9)
    A3, lo3, hi3 = _rows3()
    xlo, xhi = [0.0] * 9, [0.0] * 9
    xlo[4], xhi[4] = -0.02, 0.02
    kw = dict(x_box_mask=1 << 4, x_box_lo=tuple(xlo), x_box_hi=tuple(xhi))
    okw = dict(kw, x_row_count=3, x_row_a=tuple(A3.reshape(-1)) + (0.0,) * 54, x_row_lo=tuple(lo3) + (0.0,) * 6,
               x_row_hi=tuple(hi3) + (0.0,) * 6)
    return kw, okw, (A3, lo3, hi3), np.vstack([A3, np.eye(9)[4:5]])


def _hs_cfg(pogox=False, **over):
    import pyhostsim as hs
    from decentralized_ekf_mhe_b200.params import DekfConfig
    lib = C.CDLL(hs.build())
    cfg = DekfConfig()
    lib.hostsim_default_go1(C.byref(cfg))
    cfg.ekf_rate = 200
    if pogox:
        cfg.update(**POGOX)
    cfg.update(**over)
    return cfg


def _golden(name):
    g = np.load(GOLDEN)
    st = {k.split("/in_")[1]: g[k] for k in g.files if k.startswith(name + "/in_") and not k.endswith("_ns")}
    N, _, _, rate = (int(v) for v in g[name + "/params"])
    return st, N, rate


def _streams9():
    from decentralized_ekf_mhe_b200 import synth
    out = {"ragged_n20": (synth.to_numpy(synth.make_stream(4, 80, vo_jitter=True)), 20, 200)}
    for name in ("mhe_n5", "mhe_n5_late"):
        out[name] = _golden(name)
    return out


def oracle_joint(oracle, prm, st, inst, ticks, N, ds=9, rate=200, bound_rows=None, scale=False):
    """{T: dict(X [K][K][ds][ds][n], n_vo [n])}: the state blocks of the inverse KKT matrix of the oracle's window QP of tick T
    for the instances inst; K = min(T+1, N) (the last K states of the oracle's window).  bound_rows(T, j, K) -> [(k, a)]: rows
    a' x_k = const added as equalities (active bounds).  scale: Jacobi-scale the KKT system before the solve."""
    out = {}
    for j, i in enumerate(inst):
        ekf = oracle.Ekf(oracle.ekf_params(rate=rate))
        m = oracle.Mhe(prm)
        for s in range(max(ticks) + 1):
            vo = vq = None
            if st["vo_flag"][s, i]:
                vo = (st["vo_time_pre"][s, i], st["vo_time_now"][s, i], st["vo_rel_p"][s, :, i])
                vq = st["vo_quat"][s, :, i]
            ekf.tick(st["gyro"][s, :, i], st["accel"][s, :, i], st["imu_time"][s, i], vq, st["vo_time_now"][s, i])
            q, _ = ekf.get()
            m.step(s, imu_time=st["imu_time"][s, i], accel=st["accel"][s, :, i], gyro=st["gyro"][s, :, i], quat=q,
                   joint_pos=st["joint_pos"][s, :, i], joint_vel=st["joint_vel"][s, :, i], foot_force=st["foot_force"][s, :, i],
                   vo=vo)
            if s not in ticks:
                continue
            dsv, dm, dc, nV, _ = m.dims()
            stride = 2 * dsv + dm + dc   # var_x(j) = j (2 ds + dm + dc), oracle/mhe.c
            H, _, A, l, u = m.export_qp()
            nwin, K = min(s + 1, int(prm.N)), min(s + 1, N)
            js = list(range(nwin - K, nwin))
            rows = [A[np.abs(u - l) < 1e-9]]
            if bound_rows is not None:
                for k, a in bound_rows(s, j, K):
                    r = np.zeros((1, nV))
                    r[0, js[k] * stride:js[k] * stride + ds] = a
                    rows.append(r)
            Cm = np.vstack(rows)
            nc = Cm.shape[0]
            KKT = np.block([[H, Cm.T], [Cm, np.zeros((nc, nc))]])
            idx = np.concatenate([np.arange(p * stride, p * stride + ds) for p in js])
            E = np.zeros((KKT.shape[0], len(idx)))
            E[idx, np.arange(len(idx))] = 1.0
            if scale:
                d = np.abs(np.diag(KKT))
                sc = 1.0 / np.sqrt(np.where(d > 0, d, 1.0))
                X = sc[:, None] * np.linalg.solve(sc[:, None] * KKT * sc[None, :], sc[:, None] * E)
            else:
                X = np.linalg.solve(KKT, E)
            X = X[idx].reshape(K, ds, K, ds).transpose(0, 2, 1, 3)
            o = out.setdefault(s, dict(X=np.zeros((K, K, ds, ds, len(inst))), n_vo=np.zeros(len(inst), int)))
            o["X"][..., j] = X
            o["n_vo"][j] = (3 * (K - 1) - int((l < u).sum())) // 3 if bound_rows is None else 0
    return out


def diag_blocks(X):
    K = X.shape[0]
    return np.stack([X[k, k] for k in range(K)])


def lag_blocks(X, lag=1):
    K = X.shape[0]
    return np.stack([X[k, k + lag] for k in range(K - lag)])


def _cerr(Cm, Co, Po, free=None, lag=1):
    """max correlation-scaled error |dC_ab| / sqrt(Po_k,aa Po_k+lag,bb) of Cm [K-lag][ds][ds](...) against Co; Po [K][ds][ds](...)
    the oracle's diagonal blocks.  free [K][ds](...): the coordinates compared (None: all)."""
    d = np.sqrt(np.abs(np.einsum("kii...->ki...", Po)))
    with np.errstate(divide="ignore", invalid="ignore"):   # fixed coordinates have zero variance; `free` drops them
        e = np.abs(Cm - Co) / (d[:-lag, :, None] * d[lag:, None, :])
    if free is not None:
        e = e[free[:-lag, :, None] & free[lag:, None, :]]
    return float(e.max())


def _free_of(Po):
    """coordinates whose oracle variance is not negligible against the largest of its block (a coordinate fixed by an active
    bound has variance zero up to round-off)."""
    d = np.sqrt(np.abs(np.einsum("kii...->ki...", Po)))
    return d > 1e-6 * d.max(axis=1, keepdims=True)


def _fixed(words):
    return (words | (words >> 9)) & 0x1ff


@pytest.fixture(scope="module")
def cases9(oracle):
    out = {}
    for name, (st, N, rate) in _streams9().items():
        n = st["gyro"].shape[2]
        prm = oracle.go1_params(N=N)
        out[name] = (st, N, rate, oracle_joint(oracle, prm, st, list(range(n)), TICKS9[name], N, rate=rate))
    return out


@pytest.fixture(scope="module")
def foot_case(oracle):
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(2, FOOT_S, vo=False))
    prm = oracle.go1_params(leg_odom_type=1, N=400)
    return st, oracle_joint(oracle, prm, st, [0, 1], FOOT_TICKS, FOOT_N, ds=21, scale=True)


def _box_oracle(oracle, name, st, act, inst, ticks):
    """the constrained oracle with the bounds of the reported active words act(T, j) -> [K] as equalities."""
    kw, okw, rows, R = _kind(name)
    prm = oracle.go1_params(**POGOX, **okw)

    def bound_rows(T, j, K):
        w = act(T, j)
        return [(k, R[r]) for k in range(K) for r in range(R.shape[0]) if (int(w[k]) >> r | int(w[k]) >> (9 + r)) & 1]

    return oracle_joint(oracle, prm, st, inst, ticks, 20, bound_rows=bound_rows)


@pytest.fixture(scope="module")
def box_cases(oracle):
    import pywindowcrosssim as xs
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(3, 48, robot="pogox", vo_jitter=True))
    out = {}
    for name in ("vbox", "xbox", "rows"):
        kw, _, rows, R = _kind(name)
        r = xs.run_box(st, _hs_cfg(pogox=True, **kw), rows=rows)
        o = _box_oracle(oracle, name, st, lambda T, j: r["act"][T, :min(T + 1, 20), j], [0, 1, 2], BOX_TICKS)
        out[name] = (st, r, o, R)
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["ragged_n20", "mhe_n5", "mhe_n5_late"])
@pytest.mark.parametrize("precision", [0, 1])
def test_host_cross_matches_kkt_oracle(cases9, name, precision):
    """9-state handles, both modes: C_k within 1e-8 (fp64) / 1e-4 (fp32) of the KKT blocks (k, k+1), correlation-scaled; FULL
    equals INCREMENTAL bit for bit; the diagonal blocks of the same pass equal run_cov's bit for bit."""
    import pywindowcovsim as ws
    import pywindowcrosssim as xs
    st, N, rate, Co = cases9[name]
    assert [T for T in Co if T < N] and [T for T in Co if T >= N and (Co[T]["n_vo"] == 0).any()]
    res = []
    for mode in (0, 1):
        cfg = dict(N=N, ekf_rate=rate, window_solve=mode, precision=precision)
        r = xs.run_nine(st, _hs_cfg(**cfg))
        assert np.array_equal(r["cov"], ws.run_cov(st, _hs_cfg(**cfg))["cov"], equal_nan=True)
        err = 0.0
        for T, o in Co.items():
            K = o["X"].shape[0]
            Cm = r["cross"][T, :K - 1].reshape(K - 1, 9, 9, -1)
            assert np.isnan(r["cross"][T, K - 1:]).all()
            err = max(err, _cerr(Cm, lag_blocks(o["X"]), diag_blocks(o["X"])))
        print(f"{name} precision={precision} mode={mode}: C max correlation-scaled error {err:.3e}")
        assert err <= (TOL64 if precision == 0 else TOL32)
        res.append(r)
    assert np.array_equal(res[0]["cross"], res[1]["cross"], equal_nan=True)
    assert np.array_equal(res[0]["cov"], res[1]["cov"], equal_nan=True)


def test_host_markov_identity(cases9):
    """The window's posterior is Gauss-Markov: the KKT block (i, i+2) equals C_i P_{i+1}^-1 C_{i+1} built from the exported
    blocks (correlation-scaled, 1e-6), so the diagonal and lag-one blocks determine the whole joint posterior."""
    import pywindowcrosssim as xs
    st, N, rate, Co = cases9["ragged_n20"]
    r = xs.run_nine(st, _hs_cfg(N=N, ekf_rate=rate, window_solve=1, precision=0))
    err, cnt = 0.0, 0
    for T, o in Co.items():
        K = o["X"].shape[0]
        if K < 3:
            continue
        P = r["cov"][T, :K].reshape(K, 9, 9, -1).transpose(3, 0, 1, 2)
        Cm = r["cross"][T, :K - 1].reshape(K - 1, 9, 9, -1).transpose(3, 0, 1, 2)
        M = np.stack([Cm[:, i] @ np.linalg.solve(P[:, i + 1], Cm[:, i + 1]) for i in range(K - 2)]).transpose(0, 2, 3, 1)
        err = max(err, _cerr(M, lag_blocks(o["X"], 2), diag_blocks(o["X"]), lag=2))
        cnt += K - 2
    print(f"Markov identity over {cnt} blocks (i, i+2): max correlation-scaled error {err:.3e}")
    assert cnt > 0 and err <= 1e-6


def test_host_foot_cross_matches_exact_oracle(foot_case):
    """Foot states, the exact N = 400 oracle case: C_k within the P bar of the foot-window test (1e-6); P equals run_window's."""
    import pyfootwindowsim as fs
    import pywindowcrosssim as xs
    st, ref = foot_case
    cfg = dict(leg_odom_type=1)
    r = xs.run_foot(st, _hs_cfg(**cfg))
    assert np.array_equal(r["cov"], fs.run_window(st, _hs_cfg(**cfg))["cov"], equal_nan=True)
    err = 0.0
    for T, o in ref.items():
        K = o["X"].shape[0]
        err = max(err, _cerr(r["cross"][T, :K - 1], lag_blocks(o["X"]), diag_blocks(o["X"])))
    print(f"foot states vs exact oracle: C max correlation-scaled error {err:.3e}")
    assert err <= 1e-6


@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_host_box_cross_matches_dense_kkt(box_cases, name):
    """Constrained handles: C against the dense KKT inverse with the reported active bounds, correlation-scaled over the free
    coordinates, 1e-9; rows of components fixed at stage j and columns of those fixed at j+1 exactly 0; on rows handles
    |a_i C| and |C a_i'| <= 1e-12 scale(C) for rows active at j and j+1."""
    st, r, o, R = box_cases[name]
    err, nact = 0.0, 0
    for T, ot in o.items():
        K = ot["X"].shape[0]
        Po = diag_blocks(ot["X"])
        Cm = r["cross"][T, :K - 1]
        err = max(err, _cerr(Cm, lag_blocks(ot["X"]), Po, free=_free_of(Po)))
        fx = _fixed(r["act"][T, :K].astype(np.int64))
        nact += int((fx != 0).sum())
        for k in range(K - 1):
            for i in range(Cm.shape[-1]):
                c = Cm[k, :, :, i]
                if name != "rows":
                    rr = [a for a in range(9) if (fx[k, i] >> a) & 1]
                    cc = [a for a in range(9) if (fx[k + 1, i] >> a) & 1]
                    assert (c[rr, :] == 0).all() and (c[:, cc] == 0).all()
                else:
                    sc = np.abs(c).max() + 1e-300
                    for q in range(R.shape[0]):
                        if (fx[k, i] >> q) & 1:
                            assert np.abs(R[q] @ c).max() <= 1e-12 * sc
                        if (fx[k + 1, i] >> q) & 1:
                            assert np.abs(c @ R[q]).max() <= 1e-12 * sc
    print(f"{name}: C max correlation-scaled error {err:.3e}, {nact} states with fixed components")
    assert nact > 0 and err <= 1e-9


def test_host_box_cross_leaves_p_unchanged():
    """The serial box pass with the cross block returns the same P bit for bit; capped instances have all-NaN C blocks."""
    import pyboxwindowsim as bw
    import pywindowcrosssim as xs
    from decentralized_ekf_mhe_b200 import synth
    kw = dict(_kind("vbox")[0], v_box_max_iter=2)
    st = synth.to_numpy(synth.make_stream(24, 40, robot="pogox", vo_jitter=True))
    a = xs.run_box(st, _hs_cfg(pogox=True, **kw))
    b = bw.run_window(st, _hs_cfg(pogox=True, **kw))
    assert np.array_equal(a["cov"], b["cov"], equal_nan=True) and (a["capped"][1:] != 0).any()
    for T in range(1, 40):
        K = min(T + 1, 20)
        nan = np.isnan(a["cross"][T, :K - 1]).all(axis=(0, 1, 2))
        assert np.array_equal(nan, a["capped"][T] != 0)
        assert not np.isnan(a["cross"][T, :K - 1][..., ~nan]).any()


def _tally(name):
    exe = os.path.join(HERE, "hostsim", "_build", name)
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-o", exe, os.path.join(HERE, "hostsim", name + ".cpp")])
    return json.loads(subprocess.check_output([exe]).decode())


def test_probe_cross_flop_constants_match_tally():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import window_probe as wp
    tally = _tally("window_cross_flopcount")
    for k in ("window_cross", "box_cross", "box_rows_vcvt"):
        assert wp.FLOPS_CROSS[k] == tally[k], k
    for L in (1, 2, 4):
        assert wp.foot_stage_flops(L)["cross"] == tally["foot"][str(L)], L


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def E():
    import torch
    from decentralized_ekf_mhe_b200 import build, estimator
    build.build()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return estimator


def _est9(E, n, precision="fp64", mode=1, N=20, **over):
    return E.BatchedEstimator(E.robot_params("go1", ekf_rate=200, N=N, window_solve=mode, **over), n, precision=precision)


def _est_foot(E, n, robot="go1"):
    return E.BatchedEstimator(E.robot_params(robot, ekf_rate=200, N=FOOT_N, leg_odom_type=1), n, precision="fp64")


def _est_box(E, name, n, precision="fp64", **over):
    kw, _, rows, _ = _kind(name)
    est = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200, **kw, **over), n, precision=precision)
    if rows is not None:
        est.add_state_rows(*rows)
    return est


def _dev(st):
    import torch
    return {k: torch.as_tensor(v).cuda().contiguous() for k, v in st.items()}


def _raw(est, want_P=True, want_C=True):
    """dekf_get_window_cross_cov through ctypes: (rc, P [K][ds][ds][n] or None, C [K-1][ds][ds][n] or None, K)."""
    import torch
    h = est._hd
    N, ds, n = int(h.cfg.N), h.ds, h.n
    P = torch.full((N, ds, ds, n), -1.0, dtype=torch.float64, device="cuda") if want_P else None
    Cc = torch.full((N - 1, ds, ds, n), -1.0, dtype=torch.float64, device="cuda") if want_C else None
    K = C.c_int32(-7)
    rc = h.L.dekf_get_window_cross_cov(h.h, C.c_void_p(P.data_ptr()) if want_P else None,
                                       C.c_void_p(Cc.data_ptr()) if want_C else None, C.byref(K))
    k = K.value
    return rc, (P[:k] if want_P and rc == 0 else None), (Cc[:k - 1] if want_C and rc == 0 else None), k


def _embed(st, n, sel, robot="go1", vo=True):
    from decentralized_ekf_mhe_b200 import synth
    S = st["gyro"].shape[0]
    base = synth.to_numpy(synth.make_stream(n, S, robot=robot, vo=vo, vo_jitter=True))
    for k, v in st.items():
        base[k] = base[k].copy()
        base[k][..., sel] = v
    return base


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_device_cross_matches_kkt_oracle_9state(E, oracle, precision):
    """8 instances of a 300-instance ragged stream at the sampled ticks, both modes; FULL == INCREMENTAL bit for bit."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, N, n, ticks = 80, 20, 300, TICKS9["ragged_n20"]
    sel = np.linspace(0, n - 1, 8).astype(int)
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    idx = torch.as_tensor(sel, device="cuda")
    st = synth.to_numpy({k: v[..., idx] for k, v in d.items()})
    Co = oracle_joint(oracle, oracle.go1_params(N=N), st, list(range(len(sel))), ticks, N)
    full, incr = _est9(E, n, precision, 0), _est9(E, n, precision, 1)
    err = 0.0
    for s in range(S):
        store = E.robot_store.from_stream(d, s)
        full.step(s, store)
        incr.step(s, store)
        if s in Co:
            cf, ci = full.window_cross_cov(), incr.window_cross_cov()
            assert cf.shape == (min(s + 1, N) - 1, 9, 9, n) and torch.equal(cf, ci)
            X = Co[s]["X"]
            err = max(err, _cerr(cf[..., idx].cpu().numpy(), lag_blocks(X), diag_blocks(X)))
    print(f"9-state {precision}: device C vs oracle {err:.3e}")
    assert err <= (TOL64 if precision == "fp64" else TOL32)


@pytest.mark.gpu
def test_device_cross_matches_oracle_foot(E, foot_case):
    st, ref = foot_case
    n, sel = 300, [7, 299]
    d = _dev(_embed(st, n, sel, vo=False))
    est = _est_foot(E, n)
    err = 0.0
    for s in range(max(FOOT_TICKS) + 1):
        est.step(s, E.robot_store.from_stream(d, s))
        if s in ref:
            Cm = est.window_cross_cov()[..., sel].cpu().numpy()
            X = ref[s]["X"]
            err = max(err, _cerr(Cm, lag_blocks(X), diag_blocks(X)))
    print(f"foot states: device C vs exact oracle {err:.3e}")
    assert err <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_device_cross_matches_host_and_oracle_box(E, oracle, name):
    """fp64 constrained handles: C against the oracle (1e-8, the device P bar) and the host build (1e-9), masks exactly 0."""
    import pywindowcrosssim as xs
    from decentralized_ekf_mhe_b200 import synth
    kw, _, rows, R = _kind(name)
    S, n, m = 34, 300, 6
    st = synth.to_numpy(synth.make_stream(n, S, robot="pogox", vo_jitter=True))
    d = _dev(st)
    est = _est_box(E, name, n)
    got = {}
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
        if s in (1, 12, 20, 33):
            P, Cm = est.window_cross_cov(return_cov=True)
            got[s] = (P.cpu().numpy(), Cm.cpu().numpy(), est.window_active().cpu().numpy())
    sub = {k: np.ascontiguousarray(v[..., :m]) for k, v in st.items()}
    hres = xs.run_box(sub, _hs_cfg(pogox=True, **kw), rows=rows)
    o = _box_oracle(oracle, name, sub, lambda T, j: got[T][2][:, j], list(range(m)), tuple(got))
    eo = eh = 0.0
    for T, (P, Cm, a) in got.items():
        K = min(T + 1, 20)
        X = o[T]["X"]
        Po = diag_blocks(X)
        eo = max(eo, _cerr(Cm[..., :m], lag_blocks(X), Po, free=_free_of(Po)))
        eh = max(eh, _cerr(Cm[..., :m], hres["cross"][T, :K - 1], Po, free=_free_of(Po)))
        if name != "rows":
            fx = _fixed(a.astype(np.int64))
            for k in range(K - 1):
                for q in range(9):
                    assert (Cm[k, q, :, (fx[k] >> q) & 1 == 1] == 0).all()
                    assert (Cm[k, :, q, (fx[k + 1] >> q) & 1 == 1] == 0).all()
    print(f"{name}: device C vs oracle {eo:.3e}, vs host build {eh:.3e}")
    assert eo <= 1e-8 and eh <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("mode", [0, 1])
def test_device_cross_agrees_with_host_build_9state(E, precision, mode):
    """The bars of the covariance test's device-vs-host comparison: fp64 1e-12, fp32 1e-5 (correlation-scaled)."""
    import pywindowcrosssim as xs
    from decentralized_ekf_mhe_b200 import synth
    S = 100
    st = synth.to_numpy(synth.make_stream(64, S, vo_jitter=True))
    r = xs.run_nine(st, _hs_cfg(window_solve=mode, precision=precision))
    est = _est9(E, 64, ("fp64", "fp32")[precision], mode)
    d = _dev(st)
    err = 0.0
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
        if s >= 1:
            Cm = est.window_cross_cov().cpu().numpy()
            K = Cm.shape[0] + 1
            err = max(err, _cerr(Cm, r["cross"][s, :K - 1].reshape(K - 1, 9, 9, -1), r["cov"][s, :K].reshape(K, 9, 9, -1)))
    print(f"precision={precision} mode={mode}: device vs host build {err:.3e}")
    assert err <= (1e-12 if precision == 0 else 1e-5)


@pytest.mark.gpu
def test_device_cross_agrees_with_host_build_foot(E):
    """The bar of the foot-window test's device-vs-host comparison of P: 1e-9 (correlation-scaled)."""
    import pywindowcrosssim as xs
    from decentralized_ekf_mhe_b200 import synth
    S, n = 60, 64
    st = synth.to_numpy(synth.make_stream(n, S, vo_jitter=True))
    r = xs.run_foot(st, _hs_cfg(leg_odom_type=1))
    est = _est_foot(E, n)
    d = _dev(st)
    err = 0.0
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
        if s >= 1:
            Cm = est.window_cross_cov().cpu().numpy()
            K = Cm.shape[0] + 1
            err = max(err, _cerr(Cm, r["cross"][s, :K - 1], r["cov"][s, :K]))
    print(f"foot states: device vs host build {err:.3e}")
    assert err <= 1e-9


def _kinds():
    return [("9", "fp64", 0), ("9", "fp64", 1), ("9", "fp32", 0), ("9", "fp32", 1), ("foot", "fp64", 1),
            ("vbox", "fp64", 0), ("vbox_serial", "fp64", 0), ("xbox", "fp64", 0), ("rows", "fp64", 0), ("vbox", "fp32", 0)]


def _make(E, kind, precision, mode, n, monkeypatch=None):
    if kind == "9":
        return _est9(E, n, precision, mode)
    if kind == "foot":
        return _est_foot(E, n)
    if kind == "vbox_serial":
        monkeypatch.setenv("DEKF_BOX_SERIAL", "1")
        est = _est_box(E, "vbox", n, precision)
        monkeypatch.delenv("DEKF_BOX_SERIAL")
        return est
    return _est_box(E, kind, n, precision)


def _stream_for(kind, n, S):
    from decentralized_ekf_mhe_b200 import synth
    robot = "go1" if kind in ("9", "foot") else "pogox"
    return {k: v.contiguous() for k, v in synth.make_stream(n, S, robot=robot, vo_jitter=True, device="cuda").items()}


def _cov_getter(est, kind):
    return est.window_cov()   # dispatches to the kind's covariance getter


@pytest.mark.gpu
@pytest.mark.parametrize("kind,precision,mode", _kinds())
def test_p_of_new_call_equals_cov_getter(E, monkeypatch, kind, precision, mode):
    """P of dekf_get_window_cross_cov is the kind's covariance getter bit for bit; C-only equals C of the P + C call."""
    import torch
    n, S = 1003, 30
    d = _stream_for(kind, n, S)
    est = _make(E, kind, precision, mode, n, monkeypatch)
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
        if s in (1, 7, 19, 20, 29):
            rc, P, Cm, K = _raw(est)
            assert rc == 0 and K == min(s + 1, 20)
            Pg = _cov_getter(est, kind)
            assert torch.equal(P.nan_to_num(7.0), Pg.nan_to_num(7.0)) and torch.equal(P.isnan(), Pg.isnan()), s
            rc, _, C1, _ = _raw(est, want_P=False)
            assert rc == 0 and torch.equal(C1.nan_to_num(7.0), Cm.nan_to_num(7.0)) and torch.equal(C1.isnan(), Cm.isnan()), s
            P2, C2 = est.window_cross_cov(return_cov=True)
            assert torch.equal(P2.nan_to_num(7.0), P.nan_to_num(7.0)) and torch.equal(C2.nan_to_num(7.0), Cm.nan_to_num(7.0))
    est.close()


def _joint_psd(P, Cm, fixed=None):
    """worst Cholesky outcome of the 2x2 joint blocks [[P_k, C_k], [C_k', P_k+1]] over [K-1][n] (fixed components -- zero rows
    and columns -- replaced by unit diagonal, which removes them), with a relative jitter of 1e-12: number of failures."""
    import torch
    K, ds, n = P.shape[0], P.shape[1], P.shape[3]
    Pt = P.permute(0, 3, 1, 2)
    Ct = Cm.permute(0, 3, 1, 2)
    J = torch.cat([torch.cat([Pt[:-1], Ct], 3), torch.cat([Ct.transpose(2, 3), Pt[1:]], 3)], 2)
    if fixed is not None:
        f = torch.cat([fixed[:-1], fixed[1:]], 2).to(torch.float64)   # [K-1][n][2 ds]
        J = J + torch.diag_embed(f)
    scale = J.diagonal(dim1=2, dim2=3).abs().amax(2)
    J = J + 1e-12 * scale[..., None, None] * torch.eye(2 * ds, dtype=J.dtype, device=J.device)
    _, info = torch.linalg.cholesky_ex(J)
    return int((info != 0).sum())


@pytest.mark.gpu
def test_invariants_at_size_go1(E):
    """Go1 fp64 incremental, 65,536 instances: every joint block PSD, no NaN."""
    import torch
    n, S = 65536, 40
    d = _stream_for("9", n, S)
    est = _est9(E, n)
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
    P, Cm = est.window_cross_cov(return_cov=True)
    assert not torch.isnan(P).any() and not torch.isnan(Cm).any()
    bad = sum(_joint_psd(P[:, :, :, j:j + 8192], Cm[:, :, :, j:j + 8192]) for j in range(0, n, 8192))
    print(f"Go1 65536: {bad} joint blocks fail Cholesky")
    assert bad == 0


@pytest.mark.gpu
def test_invariants_at_size_pogox_vbox(E):
    """PogoX velocity box (config 4, team layout), 16,384 instances: joint blocks PSD after the fixed components are removed;
    NaN exactly on capped instances."""
    import torch
    n, S = 16384, 40
    d = _stream_for("vbox", n, S)
    est = _est_box(E, "vbox", n)
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
    P, Cm = est.window_cross_cov(return_cov=True)
    capped = (est.status_ & 64) != 0
    assert torch.isnan(Cm[..., capped]).all() and not torch.isnan(Cm[..., ~capped]).any()
    act = est.window_active()
    fx = (act | (act >> 9)) & 0x1ff
    fixed = torch.stack([(fx >> a) & 1 for a in range(9)], 2)   # [K][n][9]
    keep = ~capped
    bad = _joint_psd(P[..., keep], Cm[..., keep], fixed[:, keep])
    print(f"PogoX vbox 16384: {bad} joint blocks fail Cholesky, {int(capped.sum())} capped")
    assert bad == 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mode", [("9", 0), ("9", 1), ("foot", 1), ("vbox", 0), ("rows", 0)])
def test_getter_changes_no_output_and_run_equals_steps(E, kind, mode):
    """Calling the getter between ticks changes no later output; dekf_run followed by the getter equals single steps."""
    import torch
    n, S = 512, 30
    d = _stream_for(kind, n, S)
    vo = [bool(d["vo_flag"][s].any()) for s in range(S)]
    a, b = _make(E, kind, "fp64", mode, n), _make(E, kind, "fp64", mode, n)
    for s in range(S):
        store = E.robot_store.from_stream(d, s)
        a.step(s, store)
        b.step(s, store)
        if s >= 1:
            a.window_cross_cov(return_cov=True)
            a.window_cross_cov()
        for k in ("x_MHE_", "v_MHE_b_", "status_"):
            ta, tb = getattr(a, k), getattr(b, k)
            assert torch.equal(ta.nan_to_num(7.0), tb.nan_to_num(7.0)) and torch.equal(ta.isnan(), tb.isnan()), (s, k)
    ca = a.window_cross_cov()
    assert torch.equal(ca.nan_to_num(7.0), b.window_cross_cov().nan_to_num(7.0))
    r = _make(E, kind, "fp64", mode, n)
    r.run(0, S, d, vo)
    cr = r.window_cross_cov()
    assert torch.equal(cr.nan_to_num(7.0), ca.nan_to_num(7.0)) and torch.equal(cr.isnan(), ca.isnan())
    for e in (a, b, r):
        e.close()


@pytest.mark.gpu
def test_error_paths_and_reset(E):
    """Null C and est_type 1: DEKF_EINVAL; before update(T >= 1) and after dekf_reset: DEKF_ESTATE; for every kind."""
    n = 64
    kf = _est9(E, n, est_type=1)
    d = _stream_for("9", n, 6)
    for s in range(4):
        kf.step(s, E.robot_store.from_stream(d, s))
    assert _raw(kf)[0] == EINVAL and "est_type 1" in kf._hd.L.dekf_last_error(kf._hd.h).decode()
    kf.close()
    for kind in ("9", "foot", "vbox", "rows"):
        d = _stream_for(kind, n, 6)
        est = _make(E, kind, "fp64", 1, n)
        assert _raw(est)[0] == ESTATE
        est.step(0, E.robot_store.from_stream(d, 0))
        assert _raw(est)[0] == ESTATE
        est.step(1, E.robot_store.from_stream(d, 1))
        assert _raw(est, want_C=False)[0] == EINVAL
        rc, _, _, K = _raw(est)
        assert rc == 0 and K == 2
        assert est._hd.L.dekf_reset(est._hd.h) == 0
        assert _raw(est)[0] == ESTATE
        est.close()


_FACADE_MAIN = r"""
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <vector>
#include "dekf_b200/DecentralEst.hpp"
static void rd(std::FILE *f, void *p, size_t bytes) { if (std::fread(p, 1, bytes, f) != bytes) std::exit(2); }
int main(int, char **argv) {
  std::FILE *f = std::fopen(argv[1], "rb");
  int32_t hdr[4];
  rd(f, hdr, sizeof(hdr));
  const int S = hdr[0], n = hdr[1], nq = hdr[2], nl = hdr[3];
  auto params = std::make_shared<dekf::robot_params>(dekf::robot_params::go1());
  params->n_instances_ = n;
  auto store = std::make_shared<dekf::robot_store>();
  store->resize(n, nq, nl);
  dekf::DecentralizedEstimation mhe;
  for (int T = 0; T < S; ++T) {
    rd(f, store->angular_b_.data(), sizeof(double) * 3 * n);
    rd(f, store->accel_b_.data(), sizeof(double) * 3 * n);
    rd(f, store->imu_time_.data(), sizeof(double) * n);
    rd(f, store->joint_states_position_.data(), sizeof(double) * (size_t)nq * n);
    rd(f, store->joint_states_velocity_.data(), sizeof(double) * (size_t)nq * n);
    rd(f, store->joint_states_position_.data() + (size_t)nq * n, sizeof(double) * (size_t)nl * n);
    rd(f, store->vo_new_.data(), n);
    rd(f, store->vo_time_pre_.data(), sizeof(double) * n);
    rd(f, store->vo_time_now_.data(), sizeof(double) * n);
    rd(f, store->vo_p_body_pre_2_body_.data(), sizeof(double) * 3 * n);
    rd(f, store->quaternion_.data(), sizeof(double) * 4 * n);
    if (T == 0) mhe.initialize(store, params); else mhe.update(T);
  }
  const std::vector<double> Cc = mhe.mhe_qp_.P_window_cross();
  std::FILE *o = std::fopen(argv[2], "wb");
  std::fwrite(Cc.data(), sizeof(double), Cc.size(), o);
  std::fclose(o);
  return 0;
}
"""


@pytest.mark.gpu
def test_mirrors_equal_device_getter(E, tmp_path):
    """Selector 16, BatchedEstimator.window_cross_cov(), mhe_qp_.P_window_cross() and the C++ facade's
    mhe_qp_.P_window_cross() return the device getter's blocks bit for bit (and selector 16 on a foot and a box handle)."""
    import torch
    from decentralized_ekf_mhe_b200 import build, synth
    n, S = 48, 60
    st = synth.to_numpy(synth.make_stream(n, S, vo_jitter=True))
    nq, nl = st["joint_pos"].shape[1], st["foot_force"].shape[1]
    quat = np.tile(np.array([1.0, 0.0, 0.0, 0.0])[None, :, None], (S, 1, n)) + 0.01 * np.sin(st["imu_time"])[:, None, :]
    quat /= np.linalg.norm(quat, axis=1, keepdims=True)
    d = _dev(st)
    prm = E.robot_params("go1")
    mhe = E.DecentralizedEstimation(n)
    store = E.robot_store()
    for s in range(S):
        snap = E.robot_store.from_stream(d, s)
        for f in E.robot_store.FIELDS:
            setattr(store, f, getattr(snap, f))
        store.quaternion_ = torch.as_tensor(quat[s]).cuda().contiguous()
        if s == 0:
            mhe.initialize(store, prm)
        else:
            mhe.update(s)
    C_dev = mhe.mhe_qp_.P_window_cross()
    assert C_dev.shape == (19, 9, 9, n)
    P2, C2 = mhe.mhe_qp_.P_window_cross(return_cov=True)
    assert torch.equal(C2, C_dev) and torch.equal(P2, mhe.mhe_qp_.P_window())
    h = mhe._hd
    C_raw = torch.empty(19, 81, n, dtype=torch.float64, device="cuda")
    K = C.c_int32()
    h.check(h.L.dekf_get_window_cross_cov(h.h, None, C.c_void_p(C_raw.data_ptr()), C.byref(K)), "dekf_get_window_cross_cov")
    assert K.value == 20 and torch.equal(C_raw.view(19, 9, 9, n), C_dev)
    host = np.zeros((19 * 81, n))
    h.check(h.L.dekf_get_host(h.h, 16, host.ctypes.data_as(C.c_void_p)), "dekf_get_host")
    assert np.array_equal(host.reshape(19, 9, 9, n), C_dev.cpu().numpy())
    be = _est9(E, n)
    for s in range(S):
        be.step(s, E.robot_store.from_stream(d, s))
    hb = be._hd
    h.check(hb.L.dekf_get_window_cross_cov(hb.h, None, C.c_void_p(C_raw.data_ptr()), None), "dekf_get_window_cross_cov")
    assert torch.equal(be.window_cross_cov(), C_raw.view(19, 9, 9, n))
    for kind in ("foot", "rows"):   # selector 16 on the other kinds
        e = _make(E, kind, "fp64", 1, n)
        dk = _stream_for(kind, n, 24)
        for s in range(24):
            e.step(s, E.robot_store.from_stream(dk, s))
        ds = e._hd.ds
        hk = np.zeros((19 * ds * ds, n))
        assert e._hd.L.dekf_get_host(e._hd.h, 16, hk.ctypes.data_as(C.c_void_p)) == 0
        assert np.array_equal(hk.reshape(19, ds, ds, n), e.window_cross_cov().cpu().numpy(), equal_nan=True)
        e.close()
    so = build.build()
    src, exe = tmp_path / "cross_main.cpp", str(tmp_path / "cross_main")
    src.write_text(_FACADE_MAIN)
    libdir = os.path.dirname(so)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe, "-L", libdir,
                           "-ldekf_b200", f"-Wl,-rpath,{libdir}"])
    path, outp = str(tmp_path / "stream.bin"), str(tmp_path / "out.bin")
    with open(path, "wb") as f:
        f.write(np.array([S, n, nq, nl], np.int32).tobytes())
        for s in range(S):
            for k in ("gyro", "accel", "imu_time", "joint_pos", "joint_vel", "foot_force"):
                f.write(np.ascontiguousarray(st[k][s], np.float64).tobytes())
            f.write(np.ascontiguousarray(st["vo_flag"][s], np.uint8).tobytes())
            for k in ("vo_time_pre", "vo_time_now", "vo_rel_p"):
                f.write(np.ascontiguousarray(st[k][s], np.float64).tobytes())
            f.write(np.ascontiguousarray(quat[s], np.float64).tobytes())
    r = subprocess.run([exe, path, outp], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    C_cpp = np.fromfile(outp, np.float64)
    assert C_cpp.size == 19 * 81 * n and np.array_equal(C_cpp.reshape(19, 9, 9, n), C_dev.cpu().numpy())
