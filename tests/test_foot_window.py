"""Smoothed window of the foot-position-state model (leg_odom_type 1, dekf_get_foot_window): the optimum of every window
state over all ds = 9 + 3L components and its ds x ds posterior covariance, by a backward pass over the factors of the step's
information-form sweep (csrc/footstate.cuh foot_window_smooth, csrc/foot_window.cuh).

Oracles:
- exact: oracle.Mhe with N = 400 on a stream without VO never marginalises, so its full-history optimum (solution()) and the
  x_k blocks of its inverse KKT matrix (export_qp()), restricted to the last K states, are the window's exact answer.  The KKT
  system is Jacobi-scaled before the solve because the foot weights span about 4e-10 .. 4e10; its residual is checked.
- literal: N = 20 on ragged-VO streams, with the known 1e-5 noise floor of its marginalisation on the feet.
CPU: the host build (tests/hostsim/foot_window_hostsim.cpp).  GPU (-m gpu): the device getter against both oracles and the
host build, bit-identity of row K-1 with dekf_outputs.x, output invariance, the pipelined run, the other robots, the error
paths and the host-side mirrors."""
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
N = 20
EXACT_S, EXACT_TICKS, EXACT_COV_TICKS = 46, (3, 12, 19, 20, 21, 33, 45), (12, 20, 33, 45)
LIT_S, LIT_TICKS = 70, (4, 15, 19, 20, 21, 37, 52, 69)


def _hs_cfg(**over):
    import pyhostsim as hs
    from decentralized_ekf_mhe_b200.params import DekfConfig
    lib = C.CDLL(hs.build())
    cfg = DekfConfig()
    lib.hostsim_default_go1(C.byref(cfg))
    cfg.ekf_rate = 200
    cfg.leg_odom_type = 1
    cfg.update(**over)
    return cfg


def _step_oracle(oracle, st, i, prm, ticks, cov_ticks=()):
    """{T: (x [K][ds], P [K][ds][ds] or None, KKT residual)} for instance i at the given ticks; K = min(T+1, N)."""
    out = {}
    ekf = oracle.Ekf(oracle.ekf_params(rate=200))
    m = oracle.Mhe(prm)
    for s in range(max(ticks) + 1):
        vo = vq = None
        if st["vo_flag"][s, i]:
            vo = (st["vo_time_pre"][s, i], st["vo_time_now"][s, i], st["vo_rel_p"][s, :, i])
            vq = st["vo_quat"][s, :, i]
        ekf.tick(st["gyro"][s, :, i], st["accel"][s, :, i], st["imu_time"][s, i], vq, st["vo_time_now"][s, i])
        q, _ = ekf.get()
        m.step(s, imu_time=st["imu_time"][s, i], accel=st["accel"][s, :, i], gyro=st["gyro"][s, :, i], quat=q,
               joint_pos=st["joint_pos"][s, :, i], joint_vel=st["joint_vel"][s, :, i], foot_force=st["foot_force"][s, :, i], vo=vo)
        if s not in ticks:
            continue
        ds, dm, dc, _, _ = m.dims()
        stride = 2 * ds + dm + dc   # var_x(j) = j (2 ds + dm + dc), oracle/mhe.c
        sol = m.solution()
        nwin = min(s + 1, int(prm.N))          # states the oracle's window holds
        K = min(s + 1, N)
        js = range(nwin - K, nwin)
        x = np.array([sol[j * stride:j * stride + ds] for j in js])
        P, res = None, 0.0
        if s in cov_ticks:
            H, _, A, l, u = m.export_qp()
            Ae = A[l == u]
            ne = Ae.shape[0]
            KKT = np.block([[H, Ae.T], [Ae, np.zeros((ne, ne))]])
            idx = np.concatenate([np.arange(j * stride, j * stride + ds) for j in js])
            d = np.abs(np.diag(KKT))
            sc = 1.0 / np.sqrt(np.where(d > 0, d, 1.0))
            E = np.zeros((KKT.shape[0], len(idx)))
            E[idx, np.arange(len(idx))] = 1.0
            Z = np.linalg.solve(sc[:, None] * KKT * sc[None, :], sc[:, None] * E)
            X = sc[:, None] * Z
            res = float(np.abs(KKT @ X - E).max() / np.abs(KKT).max())
            X = X[idx]
            P = np.array([X[ds * k:ds * k + ds, ds * k:ds * k + ds] for k in range(K)])
        out[s] = (x, P, res)
    return out


def cov_error(P, Po):
    """max correlation-scaled error |dP_ij| / sqrt(Po_ii Po_jj) over [K][ds][ds] (and any trailing instance axis)."""
    d = np.sqrt(np.einsum("kii...->ki...", Po))
    return float((np.abs(P - Po) / (d[:, :, None] * d[:, None, :])).max())


@pytest.fixture(scope="module")
def exact_case(oracle):
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(2, EXACT_S, vo=False))
    prm = oracle.go1_params(leg_odom_type=1, N=400)
    ref = [_step_oracle(oracle, st, i, prm, EXACT_TICKS, EXACT_COV_TICKS) for i in range(2)]
    return st, ref


@pytest.fixture(scope="module")
def literal_case(oracle):
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(2, LIT_S, vo_jitter=True))
    prm = oracle.go1_params(leg_odom_type=1)
    assert int(prm.N) == N
    ref = [_step_oracle(oracle, st, i, prm, LIT_TICKS) for i in range(2)]
    return st, ref


def _coverage(ticks):
    assert any(T < N for T in ticks) and N in ticks and any(T > N for T in ticks)


def exact_errors(win, cov, ref, ticks, cov_ticks):
    """(max |dx|, max correlation-scaled dP, max oracle residual) of win [S][N][ds][n] / cov [S][N][ds][ds][n]."""
    ex = ep = rs = 0.0
    for i, r in enumerate(ref):
        for T in ticks:
            xo, Po, res = r[T]
            K = xo.shape[0]
            ex = max(ex, float(np.abs(win[T][:K, :, i] - xo).max()))
            if T in cov_ticks:
                ep = max(ep, cov_error(cov[T][:K, :, :, i], Po))
                rs = max(rs, res)
    return ex, ep, rs


def literal_errors(win, ref, ticks):
    """(base states, feet, all components at T < N) max errors."""
    eb = ef = es = 0.0
    for i, r in enumerate(ref):
        for T in ticks:
            xo = r[T][0]
            K = xo.shape[0]
            d = np.abs(win[T][:K, :, i] - xo)
            eb, ef = max(eb, float(d[:, :9].max())), max(ef, float(d[:, 9:].max()))
            if T < N:
                es = max(es, float(d.max()))
    return eb, ef, es


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_host_window_matches_exact_oracle(exact_case):
    import pyfootwindowsim as fs
    st, ref = exact_case
    _coverage(EXACT_TICKS)
    r = fs.run_window(st, _hs_cfg())
    ex, ep, rs = exact_errors(r["win"], r["cov"], ref, EXACT_TICKS, EXACT_COV_TICKS)
    print(f"host vs exact oracle: x {ex:.3e}, P (correlation-scaled) {ep:.3e}, oracle KKT residual {rs:.3e}")
    assert rs < 1e-9
    assert ex <= 1e-8 and ep <= 1e-6


def test_host_window_matches_literal_oracle(literal_case):
    import pyfootwindowsim as fs
    st, ref = literal_case
    _coverage(LIT_TICKS)
    assert st["vo_flag"].any()
    r = fs.run_window(st, _hs_cfg())
    eb, ef, es = literal_errors(r["win"], ref, LIT_TICKS)
    print(f"host vs literal oracle: base {eb:.3e}, feet {ef:.3e}, T < N {es:.3e}")
    assert eb <= 1e-6 and ef <= 1e-5 and es <= 1e-8


def test_host_window_invariants():
    """Row K-1 == foot_solve's x_T bit for bit; every block exactly symmetric and positive definite; block K-1 == M_T^-1."""
    import pyfootwindowsim as fs
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(4, 50, vo_jitter=True))
    r = fs.run_window(st, _hs_cfg())
    worst = 0.0
    for s in range(1, 50):
        K = min(s + 1, N)
        assert np.array_equal(r["win"][s, K - 1], r["x"][s])
        assert np.isnan(r["win"][s, K:]).all()
        P = r["cov"][s, :K]
        assert np.array_equal(P, P.transpose(0, 2, 1, 3))
        np.linalg.cholesky(P.transpose(0, 3, 1, 2))
        Pinv = np.linalg.inv(r["info"][s].transpose(2, 0, 1)).transpose(1, 2, 0)
        worst = max(worst, cov_error(P[K - 1][None], Pinv[None]))
    print(f"block K-1 vs inverse information matrix: {worst:.3e}")
    assert worst <= 1e-12


def _tally():
    src = os.path.join(HERE, "hostsim", "foot_window_flopcount.cpp")
    out = os.path.join(HERE, "hostsim", "_build", "foot_window_flopcount")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", out, src])
    return json.loads(subprocess.check_output([out]).decode())


def test_probe_foot_flop_closed_form_matches_tally():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import window_probe
    tally = _tally()
    for L in (1, 2, 4):
        got = window_probe.foot_stage_flops(L)
        for k in ("mean", "cov", "cov_T"):
            assert got[k] == tally[str(L)][k], (L, k, got[k], tally[str(L)][k])


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def est_mod():
    import torch
    from decentralized_ekf_mhe_b200 import build, estimator
    build.build()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return estimator


def _est(estimator, n, robot="go1", **over):
    prm = estimator.robot_params(robot, ekf_rate=200, N=N, leg_odom_type=1, **over)
    return estimator.BatchedEstimator(prm, n, precision="fp64")


def _dev(st):
    import torch
    return {k: torch.as_tensor(v).cuda().contiguous() for k, v in st.items()}


def _getter(est, want_x=True, want_P=True):
    import torch
    h = est._hd
    x = torch.empty(N, h.ds, h.n, dtype=torch.float64, device="cuda") if want_x else None
    P = torch.empty(N, h.ds * h.ds, h.n, dtype=torch.float64, device="cuda") if want_P else None
    K = C.c_int32()
    rc = h.L.dekf_get_foot_window(h.h, C.c_void_p(x.data_ptr()) if want_x else None, C.c_void_p(P.data_ptr()) if want_P else None,
                                  C.byref(K))
    h.check(rc, "dekf_get_foot_window")
    k = K.value
    return (x[:k] if want_x else None), (P[:k].view(k, h.ds, h.ds, h.n) if want_P else None)


def _embed(st, n, sel):
    """the instances of st placed at columns sel of an n-instance stream (the others: synthetic filler)."""
    from decentralized_ekf_mhe_b200 import synth
    S = st["gyro"].shape[0]
    base = synth.to_numpy(synth.make_stream(n, S, vo=bool(st["vo_flag"].any()), vo_jitter=True))
    for k, v in st.items():
        base[k] = base[k].copy()
        base[k][..., sel] = v
    return base


@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 1003])
def test_device_window_matches_oracles(est_mod, exact_case, literal_case, n):
    sel = [7, n - 1]
    for name, (st, ref), ticks, cov_ticks in (("exact", exact_case, EXACT_TICKS, EXACT_COV_TICKS),
                                              ("literal", literal_case, LIT_TICKS, ())):
        big = _embed(st, n, sel)
        d = _dev(big)
        est = _est(est_mod, n)
        win, cov = {}, {}
        for s in range(max(ticks) + 1):
            est.step(s, est_mod.robot_store.from_stream(d, s))
            if s in ticks:
                x, P = _getter(est)
                win[s] = x[..., sel].cpu().numpy()
                cov[s] = P[..., sel].cpu().numpy()
        if name == "exact":
            ex, ep, _ = exact_errors(win, cov, ref, ticks, cov_ticks)
            print(f"n={n} device vs exact oracle: x {ex:.3e}, P {ep:.3e}")
            assert ex <= 1e-8 and ep <= 1e-6
        else:
            eb, ef, es = literal_errors(win, ref, ticks)
            print(f"n={n} device vs literal oracle: base {eb:.3e}, feet {ef:.3e}, T < N {es:.3e}")
            assert eb <= 1e-6 and ef <= 1e-5 and es <= 1e-8


@pytest.mark.gpu
def test_last_row_is_outputs_x(est_mod, monkeypatch):
    """Row K-1 == dekf_outputs.x bit for bit at every tick on default (team) handles; within the team-vs-serial bars on
    DEKF_FOOT_SERIAL=1 handles; x-only, P-only and x+P calls agree bit for bit."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 60, 1003
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    est = _est(est_mod, n)
    monkeypatch.setenv("DEKF_FOOT_SERIAL", "1")
    ser = _est(est_mod, n)
    monkeypatch.delenv("DEKF_FOOT_SERIAL")
    wb = wf = 0.0
    for s in range(S):
        store = est_mod.robot_store.from_stream(d, s)
        est.step(s, store)
        ser.step(s, store)
        if s < 1:
            continue
        x, P = _getter(est)
        assert torch.equal(x[-1], est.x_MHE_), s
        x1, _ = _getter(est, want_P=False)
        _, P1 = _getter(est, want_x=False)
        assert torch.equal(x1, x) and torch.equal(P1, P), s
        xs, _ = _getter(ser, want_P=False)
        dx = (xs[-1] - ser.x_MHE_).abs()
        wb, wf = max(wb, dx[:9].max().item()), max(wf, dx[9:].max().item())
    print(f"serial handle: row K-1 vs outputs.x base {wb:.3e}, feet {wf:.3e}")
    assert wb <= 1e-9 and wf <= 1e-8


@pytest.mark.gpu
def test_device_agrees_with_host_build(est_mod):
    import pyfootwindowsim as fs
    from decentralized_ekf_mhe_b200 import synth
    S, n = 60, 64
    st = synth.to_numpy(synth.make_stream(n, S, vo_jitter=True))
    r = fs.run_window(st, _hs_cfg())
    est = _est(est_mod, n)
    d = _dev(st)
    eb = ef = ep = 0.0
    for s in range(S):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        if s < 1:
            continue
        x, P = _getter(est)
        K = x.shape[0]
        dx = np.abs(x.cpu().numpy() - r["win"][s, :K])
        eb, ef = max(eb, float(dx[:, :9].max())), max(ef, float(dx[:, 9:].max()))
        ep = max(ep, cov_error(P.cpu().numpy(), r["cov"][s, :K]))
    print(f"device vs host build: base {eb:.3e}, feet {ef:.3e}, P (correlation-scaled) {ep:.3e}")
    # P: both sides are ~3e-10 (correlation-scaled) from the exact oracle, and the stage records differ in the last bits
    # (the kinematics' sin / cos round differently on the device and in the host's libm); measured 3.1e-10 on a B200
    assert eb <= 1e-9 and ef <= 1e-8 and ep <= 1e-9


@pytest.mark.gpu
def test_getter_changes_nothing_and_run_equals_steps(est_mod):
    """Two handles on the same stream, one calling the getter every tick: all outputs and later windows bit-identical.
    dekf_run followed by the getter == tick-by-tick stepping followed by the getter.  The ring is allocated once."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 50, 300
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    a, b = _est(est_mod, n), _est(est_mod, n)
    bytes0 = a.device_bytes()
    for s in range(S):
        store = est_mod.robot_store.from_stream(d, s)
        a.step(s, store)
        b.step(s, store)
        if s >= 1:
            _getter(a)
        for k in ("x_MHE_", "v_MHE_b_", "status_"):
            ta, tb = getattr(a, k), getattr(b, k)
            assert torch.equal(ta.nan_to_num(), tb.nan_to_num()) if ta.is_floating_point() else torch.equal(ta, tb), (s, k)
        if s == 1:
            grown = a.device_bytes() - bytes0
    xa, Pa = _getter(a)
    xb, Pb = _getter(b)
    assert torch.equal(xa, xb) and torch.equal(Pa, Pb)
    assert torch.equal(a.mhe_qp_.M_p, b.mhe_qp_.M_p)
    ns = (n + 127) // 128 * 128            # padded instance stride of the device arrays
    assert grown == (N - 1) * ns * (231 + 279 + 21) * 8 and a.device_bytes() == bytes0 + grown
    c = _est(est_mod, n)
    vo = [bool(d["vo_flag"][s].any()) for s in range(S)]
    c.run(0, S, d, vo)
    xc, Pc = _getter(c)
    assert torch.equal(xc, xa) and torch.equal(Pc, Pa)


@pytest.mark.gpu
@pytest.mark.parametrize("robot,legs", [("cassie", 2), ("pogox", 1)])
def test_other_robots(est_mod, robot, legs):
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 30, 200
    d = synth.make_stream(n, S, vo_jitter=True, robot=robot, device="cuda")
    est = _est(est_mod, n, robot)
    ds = 9 + 3 * legs
    for s in range(S):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        if s < 1:
            continue
        x, P = _getter(est)
        K = min(s + 1, N)
        assert x.shape == (K, ds, n) and P.shape == (K, ds, ds, n)
        assert torch.equal(x[-1], est.x_MHE_)
        assert torch.equal(P, P.transpose(1, 2))
        torch.linalg.cholesky(P.permute(0, 3, 1, 2))


@pytest.mark.gpu
def test_error_paths_and_reset(est_mod):
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 30, 128
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    buf = torch.empty(N * 21 * 21, n, dtype=torch.float64, device="cuda")

    def rc_of(est, x=True, P=False):
        h = est._hd
        rc = h.L.dekf_get_foot_window(h.h, C.c_void_p(buf.data_ptr()) if x else None, C.c_void_p(buf.data_ptr()) if P else None, None)
        return rc, h.L.dekf_last_error(h.h).decode()

    for over, needle in ((dict(est_type=1), "est_type"), (dict(leg_odom_type=0), "dekf_get_window")):
        prm = est_mod.robot_params("go1", ekf_rate=200, N=N, **{"leg_odom_type": 1, **over})
        e = est_mod.BatchedEstimator(prm, n, precision="fp64")
        for s in range(3):
            e.step(s, est_mod.robot_store.from_stream(d, s))
        rc, msg = rc_of(e)
        assert rc == -1 and msg.startswith("dekf_get_foot_window") and needle in msg, (over, rc, msg)
    e = _est(est_mod, n)
    assert rc_of(e)[0] == -5
    e.step(0, est_mod.robot_store.from_stream(d, 0))
    assert rc_of(e)[0] == -5
    e.step(1, est_mod.robot_store.from_stream(d, 1))
    assert rc_of(e, x=False, P=False)[0] == -1
    assert rc_of(e)[0] == 0
    for s in range(2, S):
        e.step(s, est_mod.robot_store.from_stream(d, s))
    e.reset()
    assert rc_of(e)[0] == -5
    for s in range(S):
        e.step(s, est_mod.robot_store.from_stream(d, s))
    fresh = _est(est_mod, n)
    for s in range(S):
        fresh.step(s, est_mod.robot_store.from_stream(d, s))
    xa, Pa = _getter(e)
    xb, Pb = _getter(fresh)
    assert torch.equal(xa, xb) and torch.equal(Pa, Pb)


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
  params->leg_odom_type_ = 1;
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
  const std::vector<double> x = mhe.mhe_qp_.x_window(), P = mhe.mhe_qp_.P_window();
  std::FILE *o = std::fopen(argv[2], "wb");
  std::fwrite(x.data(), sizeof(double), x.size(), o);
  std::fwrite(P.data(), sizeof(double), P.size(), o);
  std::fclose(o);
  return 0;
}
"""


@pytest.mark.gpu
def test_mirrors_equal_device_getter(est_mod, tmp_path):
    """dekf_get_host(11 / 12), BatchedEstimator.window() / window_cov(), DecentralizedEstimation.mhe_qp_ views and the C++
    facade all return the device getter's bits on a foot handle."""
    import torch
    from decentralized_ekf_mhe_b200 import build, synth
    n, S, ds = 48, 40, 21
    st = synth.to_numpy(synth.make_stream(n, S, vo_jitter=True))
    nq, nl = st["joint_pos"].shape[1], st["foot_force"].shape[1]
    quat = np.tile(np.array([1.0, 0.0, 0.0, 0.0])[None, :, None], (S, 1, n)) + 0.01 * np.sin(st["imu_time"])[:, None, :]
    quat /= np.linalg.norm(quat, axis=1, keepdims=True)
    d = _dev(st)
    be = _est(est_mod, n)
    for s in range(S):
        be.step(s, est_mod.robot_store.from_stream(d, s))
    x, P = _getter(be)
    assert torch.equal(be.window(), x) and torch.equal(be.window_cov(), P)
    h = be._hd
    hx = np.zeros((N * ds, n))
    h.check(h.L.dekf_get_host(h.h, 11, hx.ctypes.data_as(C.c_void_p)), "dekf_get_host")
    hP = np.zeros((N * ds * ds, n))
    h.check(h.L.dekf_get_host(h.h, 12, hP.ctypes.data_as(C.c_void_p)), "dekf_get_host")
    assert np.array_equal(hx.reshape(N, ds, n), x.cpu().numpy()) and np.array_equal(hP.reshape(N, ds, ds, n), P.cpu().numpy())
    # the reference-shaped class with host-side orientations, and the C++ facade over the same inputs
    prm = est_mod.robot_params("go1", leg_odom_type=1)
    mhe = est_mod.DecentralizedEstimation(n)
    store = est_mod.robot_store()
    for s in range(S):
        snap = est_mod.robot_store.from_stream(d, s)
        for f in est_mod.robot_store.FIELDS:
            setattr(store, f, getattr(snap, f))
        store.quaternion_ = torch.as_tensor(quat[s]).cuda().contiguous()
        if s == 0:
            mhe.initialize(store, prm)
        else:
            mhe.update(s)
    xw, Pw = mhe.mhe_qp_.x_window(), mhe.mhe_qp_.P_window()
    x2, P2 = _getter(mhe)
    assert xw.shape == (N, ds, n) and torch.equal(xw, x2) and torch.equal(Pw, P2)
    so = build.build()
    src, exe = tmp_path / "foot_main.cpp", str(tmp_path / "foot_main")
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
    out = np.fromfile(outp, np.float64)
    assert out.size == N * ds * n + N * ds * ds * n
    assert np.array_equal(out[:N * ds * n].reshape(N, ds, n), xw.cpu().numpy())
    assert np.array_equal(out[N * ds * n:].reshape(N, ds, ds, n), Pw.cpu().numpy())


@pytest.mark.gpu
def test_smoothing_beats_filtering_on_truth(est_mod):
    """Against the synthetic ground truth, the lag-10 smoothed base velocity has a lower RMS error than the filtered
    estimate of the same stage."""
    from decentralized_ekf_mhe_b200 import synth
    S, n, lag = 120, 256, 10
    d = synth.make_stream(n, S, vo_jitter=True, truth=True, device="cuda")
    est = _est(est_mod, n)
    filt, es, ef = {}, [], []
    for s in range(S):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        if s < 1:
            continue
        filt[s] = est.x_MHE_[3:6].cpu().numpy()
        x, _ = _getter(est, want_P=False)
        k = s - lag
        if s >= 40 and k in filt:
            K = x.shape[0]
            vs = x[K - 1 - lag, 3:6].cpu().numpy()
            vt = d["v_true"][k].cpu().numpy()
            es.append(((vs - vt) ** 2).mean())
            ef.append(((filt[k] - vt) ** 2).mean())
    rs, rf = float(np.sqrt(np.mean(es))), float(np.sqrt(np.mean(ef)))
    print(f"lag-{lag} base velocity RMS error: smoothed {rs:.4e}, filtered {rf:.4e}")
    assert rs < rf
