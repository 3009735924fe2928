"""Smoothed covariances of the MHE window (dekf_get_window_cov): for every window state the 9x9 block of the window QP's
posterior covariance, computed by the covariance half of the Rauch-Tung-Striebel pass (csrc/estimator_core.cuh,
mhe_window_cov).

Oracle: the oracle's window QP of the same tick (Mhe.export_qp()), its equality rows A_e, KKT = [[H, A_e'], [A_e, 0]] solved
for the unit columns of the state variables; the x_k blocks of the solution are the covariances.  Errors are correlation-scaled,
|dP_ij| / sqrt(P_ii P_jj) with the oracle's diagonal.  CPU: the kernel body compiled for the host (tests/hostsim/window_cov_hostsim.cpp).  GPU (-m gpu):
the device getter against the oracle and the host build, the pipelined run, output invariance, information monotonicity, the
error paths and the host-side mirrors."""
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
# sampled ticks per stream: T < N, T >= N without VO equalities, and T >= N with them (the test asserts the coverage)
TICKS = {"ragged_n20": (1, 6, 15, 19, 25, 33, 44, 52, 61, 79), "mhe_n5": (1, 3, 4, 9, 30, 57, 80, 119),
         "mhe_n5_late": (1, 3, 4, 12, 40, 63, 79)}


def _hs_cfg(**over):
    import pyhostsim as hs
    from decentralized_ekf_mhe_b200.params import DekfConfig
    lib = C.CDLL(hs.build())
    cfg = DekfConfig()
    lib.hostsim_default_go1(C.byref(cfg))
    cfg.ekf_rate = 200
    cfg.update(**over)
    return cfg


def _golden(name):
    g = np.load(GOLDEN)
    st = {k.split("/in_")[1]: g[k] for k in g.files if k.startswith(name + "/in_") and not k.endswith("_ns")}
    N, _, _, rate = (int(v) for v in g[name + "/params"])
    return st, N, rate


def _streams():
    from decentralized_ekf_mhe_b200 import synth
    out = {"ragged_n20": (synth.to_numpy(synth.make_stream(4, 80, vo_jitter=True)), 20, 200)}
    for name in ("mhe_n5", "mhe_n5_late"):
        out[name] = _golden(name)
    return out


def oracle_covs(oracle, st, N, rate, inst, ticks):
    """{T: (cov [K][9][9][len(inst)], VO equality rows per instance)} from the oracle's window KKT system of tick T."""
    out = {T: (np.full((min(T + 1, N), 9, 9, len(inst)), np.nan), np.zeros(len(inst), int)) for T in ticks}
    prm = oracle.go1_params(N=N)
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
            if s not in out:
                continue
            ds, dm, dc, _, _ = m.dims()
            H, _, A, l, u = m.export_qp()
            eq = l == u
            Ae = A[eq]
            ne = Ae.shape[0]
            KKT = np.block([[H, Ae.T], [Ae, np.zeros((ne, ne))]])
            K, stride = min(s + 1, N), 2 * ds + dm + dc   # var_x(j) = j (2 ds + dm + dc), oracle/mhe.c
            idx = np.concatenate([np.arange(k * stride, k * stride + 9) for k in range(K)])
            E = np.zeros((KKT.shape[0], len(idx)))
            E[idx, np.arange(len(idx))] = 1.0
            X = np.linalg.solve(KKT, E)[idx]
            for k in range(K):
                out[s][0][k, :, :, j] = X[9 * k:9 * k + 9, 9 * k:9 * k + 9]
            # free rows are the VO placeholders, 3 per stage transition; the others have become equalities
            out[s][1][j] = (3 * (K - 1) - int((l < u).sum())) // 3
    return out


def cov_error(P, Po):
    """max correlation-scaled error of P [K][9][9][n] against Po (same shape)."""
    d = np.sqrt(np.einsum("kiin->kin", Po))
    return float((np.abs(P - Po) / (d[:, :, None, :] * d[:, None, :, :])).max())


@pytest.fixture(scope="module")
def cases(oracle):
    out = {}
    for name, (st, N, rate) in _streams().items():
        n = st["gyro"].shape[2]
        out[name] = (st, N, rate, oracle_covs(oracle, st, N, rate, list(range(n)), TICKS[name]))
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["ragged_n20", "mhe_n5", "mhe_n5_late"])
@pytest.mark.parametrize("precision", [0, 1])
def test_host_cov_matches_kkt_oracle(cases, name, precision):
    """Every window state of the sampled ticks, both solve modes: fp64 <= 1e-8, fp32 <= 1e-4 (correlation-scaled)."""
    import pywindowcovsim as ws
    st, N, rate, Co = cases[name]
    T_short = [T for T in Co if T < N]
    T_novo = [T for T in Co if T >= N and (Co[T][1] == 0).any()]
    T_vo = [T for T in Co if T >= N and (Co[T][1] > 0).any()]
    assert T_short and T_novo, (T_short, T_novo)
    assert T_vo or name == "mhe_n5_late", name   # the late-VO golden input has no equality VO row at the sampled ticks
    for mode in (0, 1):
        r = ws.run_cov(st, _hs_cfg(N=N, ekf_rate=rate, window_solve=mode, precision=precision))
        err = 0.0
        for T, (Po, _) in Co.items():
            K = Po.shape[0]
            P = r["cov"][T, :K].reshape(K, 9, 9, -1)
            err = max(err, cov_error(P, Po))
        print(f"{name} precision={precision} mode={mode}: max correlation-scaled error {err:.3e}")
        assert err <= (TOL64 if precision == 0 else TOL32)


@pytest.mark.parametrize("precision", [0, 1])
def test_host_cov_invariants(precision):
    """Every block exactly symmetric and Cholesky-factorizable; block K-1 is the filtered P_T of the checkpoint ring, widened,
    bit for bit; FULL (forward sweep into the scratch ring) equals INCREMENTAL (checkpoint ring) bit for bit."""
    import pywindowcovsim as ws
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(8, 160, vo_jitter=True))
    a = ws.run_cov(st, _hs_cfg(window_solve=0, precision=precision))
    b = ws.run_cov(st, _hs_cfg(window_solve=1, precision=precision))
    Pa, Pb = a["cov"], b["cov"]
    assert np.array_equal(np.isnan(Pa), np.isnan(Pb)) and np.array_equal(Pa[~np.isnan(Pa)], Pb[~np.isnan(Pb)])
    for s in range(1, Pa.shape[0]):
        K = min(s + 1, Pa.shape[1])
        blk = Pb[s, :K].reshape(K, 9, 9, -1)
        assert np.array_equal(blk, blk.transpose(0, 2, 1, 3))
        np.linalg.cholesky(blk.transpose(0, 3, 1, 2))      # raises if a block is not positive definite
        assert np.array_equal(Pb[s, K - 1], b["filt"][s])
        assert np.isnan(Pb[s, K:]).all()


def _tally(name):
    src = os.path.join(HERE, "hostsim", name + ".cpp")
    out = os.path.join(HERE, "hostsim", "_build", name)
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", out, src])
    return json.loads(subprocess.check_output([out]).decode())


def test_probe_cov_flop_constants_match_tally():
    tally = _tally("window_cov_flopcount")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import window_probe
    for k in ("window_cov", "window_cov_vo"):
        assert window_probe.FLOPS_COV[k] == tally[k], (k, window_probe.FLOPS_COV[k], tally[k])


# ---------------------------------------------------------------------------------------------------------------- GPU
def _est(estimator, n, precision="fp64", mode=1, N=20, rate=200, **over):
    prm = estimator.robot_params("go1", ekf_rate=rate, N=N, window_solve=mode, **over)
    return estimator.BatchedEstimator(prm, n, precision=precision)


def _dev(st):
    import torch
    return {k: torch.as_tensor(v).cuda().contiguous() for k, v in st.items()}


@pytest.fixture(scope="module")
def est_mod():
    import torch
    from decentralized_ekf_mhe_b200 import build, estimator
    build.build()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return estimator


@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 5000])
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_device_cov_matches_kkt_oracle(est_mod, oracle, n, precision):
    """8 instances at the sampled ticks of an 80-tick ragged stream against the KKT oracle; FULL == INCREMENTAL bit for bit."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, N, sel, ticks = 80, 20, np.linspace(0, n - 1, 8).astype(int), TICKS["ragged_n20"]
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    idx = torch.as_tensor(sel, device="cuda")
    st = synth.to_numpy({k: v[..., idx] for k, v in d.items()})
    Co = oracle_covs(oracle, st, N, 200, list(range(len(sel))), ticks)
    assert any((Co[T][1] > 0).any() for T in ticks)
    full, incr = _est(est_mod, n, precision, 0), _est(est_mod, n, precision, 1)
    err = 0.0
    for s in range(S):
        store = est_mod.robot_store.from_stream(d, s)
        full.step(s, store)
        incr.step(s, store)
        if s in Co:
            pf, pi = full.window_cov(), incr.window_cov()
            assert pf.shape == (min(s + 1, N), 9, 9, n) and torch.equal(pf, pi)
            err = max(err, cov_error(pf[..., idx].cpu().numpy(), Co[s][0]))
    print(f"n={n} {precision}: max correlation-scaled error {err:.3e}")
    assert err <= (TOL64 if precision == "fp64" else TOL32)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("mode", [0, 1])
def test_device_cov_agrees_with_host_build(est_mod, precision, mode):
    """Device getter against the host build of the same kernel body, 64 instances x 100 ticks, correlation-scaled.  The two do
    not see bit-identical stage records (the kinematics' sin / cos round differently on the device and in the host's libm).
    fp64 <= 1e-12.  fp32: the float filtered states differ by a few float ulps, which the smoother carries; measured 1.4e-6 on a
    B200 in both modes, bar 1e-5."""
    import pywindowcovsim as ws
    from decentralized_ekf_mhe_b200 import synth
    S = 100
    st = synth.to_numpy(synth.make_stream(64, S, vo_jitter=True))
    r = ws.run_cov(st, _hs_cfg(window_solve=mode, precision=precision))
    est = _est(est_mod, 64, ("fp64", "fp32")[precision], mode)
    d = _dev(st)
    err = 0.0
    for s in range(S):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        if s >= 1:
            P = est.window_cov().cpu().numpy()
            K = P.shape[0]
            err = max(err, cov_error(P, r["cov"][s, :K].reshape(K, 9, 9, -1)))
    print(f"precision={precision} mode={mode}: device vs host build {err:.3e} (correlation-scaled)")
    assert err <= (1e-12 if precision == 0 else 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [20000, 65536])
@pytest.mark.parametrize("mode", [0, 1])
def test_run_then_cov_equals_single_steps(est_mod, n, mode):
    """dekf_run (pipelined, internal streams joined into the handle's stream) followed by the getter == single steps + getter."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S = 100
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    vo = [bool(d["vo_flag"][s].any()) for s in range(S)]
    a, b = _est(est_mod, n, "fp64", mode), _est(est_mod, n, "fp64", mode)
    a.run(0, S, d, vo)
    pa = a.window_cov()
    for s in range(S):
        b.step(s, est_mod.robot_store.from_stream(d, s))
    assert pa.shape == (20, 9, 9, n) and torch.equal(pa, b.window_cov())


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("mode", [0, 1])
def test_cov_getter_changes_no_output(est_mod, precision, mode):
    """Later ticks, x, dekf_get_window and the arrival getters are bit-identical with and without calls to the covariance getter
    (on FULL handles both getters use the same scratch ring); the ring is allocated once and counted in dekf_device_bytes."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 70, 512
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    a, b = _est(est_mod, n, precision, mode), _est(est_mod, n, precision, mode)
    bytes0 = a.device_bytes()
    for s in range(S):
        store = est_mod.robot_store.from_stream(d, s)
        a.step(s, store)
        b.step(s, store)
        for k in ("quaternion_", "x_MHE_", "v_MHE_b_", "contact_", "status_"):
            ta, tb = getattr(a, k), getattr(b, k)
            if ta.is_floating_point():  # x / v_body are NaN before the first update
                assert torch.equal(ta.isnan(), tb.isnan()) and torch.equal(ta.nan_to_num(), tb.nan_to_num()), (s, k)
            else:
                assert torch.equal(ta, tb), (s, k)
        if s < 1:
            continue
        wa = a.window()
        a.window_cov()
        assert torch.equal(a.window(), wa) and torch.equal(wa, b.window()), s
        for x, y in zip(a.mhe_qp_.arrival_cov() + (a.mhe_qp_.M_p,), b.mhe_qp_.arrival_cov() + (b.mhe_qp_.M_p,)):
            assert torch.equal(x, y), s
    # b called only dekf_get_window: the covariance getter adds no memory of its own beyond the shared scratch ring
    assert a.device_bytes() == b.device_bytes()
    if mode == 0:
        assert a.device_bytes() >= bytes0 + 20 * 54 * n * (8 if precision == "fp64" else 4)


@pytest.mark.gpu
def test_information_monotonicity(est_mod):
    """P_k^s at tick T is no larger than the filtered covariance of x_k (block K-1 at tick k): the smallest eigenvalue of the
    difference is >= -1e-12 trace, for every window state of every tick of a ragged stream."""
    from decentralized_ekf_mhe_b200 import synth
    S, n, N = 70, 128, 20
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    est = _est(est_mod, n)
    filt, worst = {}, 0.0
    for s in range(S):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        if s < 1:
            continue
        P = est.window_cov().cpu().numpy().transpose(0, 3, 1, 2)   # [K][n][9][9]
        K = P.shape[0]
        filt[s] = P[K - 1]
        for j in range(K - 1):
            k = s - K + 1 + j
            if k not in filt:
                continue
            Dlt = filt[k] - P[j]
            ev = np.linalg.eigvalsh(Dlt).min(axis=1) / np.trace(filt[k], axis1=1, axis2=2)
            worst = min(worst, float(ev.min()))
    print(f"smallest eigenvalue of P_k|k - P_k^s over trace: {worst:.3e}")
    assert worst >= -1e-12


@pytest.mark.gpu
def test_cov_error_paths_and_reset(est_mod):
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 40, 256
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")

    def rc_of(est, ptr=True):
        h = est._hd
        P = torch.empty(20, 81, n, dtype=torch.float64, device="cuda")
        rc = h.L.dekf_get_window_cov(h.h, C.c_void_p(P.data_ptr()) if ptr else None, None)
        return rc, h.L.dekf_last_error(h.h).decode()

    for over in (dict(est_type=1), dict(leg_odom_type=1), dict(v_box_enable=1, v_box_lo=(-1, -1, -1), v_box_hi=(1, 1, 1)),
                 dict(x_box_mask=1 << 3, x_box_lo=(0, 0, 0, -1, 0, 0, 0, 0, 0), x_box_hi=(0, 0, 0, 1, 0, 0, 0, 0, 0))):
        e = _est(est_mod, n, **over)
        for s in range(3):
            e.step(s, est_mod.robot_store.from_stream(d, s))
        rc, msg = rc_of(e)
        assert rc == -1 and msg.startswith("dekf_get_window_cov"), (over, rc, msg)
    e = _est(est_mod, n)
    e.add_state_rows(np.eye(9)[3:4], [-1.0], [1.0])
    for s in range(3):
        e.step(s, est_mod.robot_store.from_stream(d, s))
    assert rc_of(e)[0] == -1 and "dekf_add_state_rows" in rc_of(e)[1]
    for mode in (0, 1):
        e = _est(est_mod, n, mode=mode)
        assert rc_of(e)[0] == -5                       # before any update
        e.step(0, est_mod.robot_store.from_stream(d, 0))
        assert rc_of(e)[0] == -5                       # T = 0: no window yet
        e.step(1, est_mod.robot_store.from_stream(d, 1))
        assert rc_of(e, ptr=False)[0] == -1            # null P
        assert rc_of(e)[0] == 0
        for s in range(2, S):
            e.step(s, est_mod.robot_store.from_stream(d, s))
        e.reset()
        assert rc_of(e)[0] == -5                       # after dekf_reset
        for s in range(S):
            e.step(s, est_mod.robot_store.from_stream(d, s))
        fresh = _est(est_mod, n, mode=mode)
        for s in range(S):
            fresh.step(s, est_mod.robot_store.from_stream(d, s))
        assert torch.equal(e.window_cov(), fresh.window_cov())


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
  const std::vector<double> P = mhe.mhe_qp_.P_window();
  std::FILE *o = std::fopen(argv[2], "wb");
  std::fwrite(P.data(), sizeof(double), P.size(), o);
  std::fclose(o);
  return 0;
}
"""


@pytest.mark.gpu
def test_cov_host_getter_python_class_api_and_cpp_facade_equal_device(est_mod, tmp_path):
    """dekf_get_host(DEKF_GET_WINDOW_P), BatchedEstimator.window_cov(), DecentralizedEstimation.mhe_qp_.P_window() and the C++
    facade's mhe_qp_.P_window() all return the device getter's covariances."""
    import torch
    from decentralized_ekf_mhe_b200 import build, synth
    n, S = 48, 60
    st = synth.to_numpy(synth.make_stream(n, S, vo_jitter=True))
    nq, nl = st["joint_pos"].shape[1], st["foot_force"].shape[1]
    quat = np.tile(np.array([1.0, 0.0, 0.0, 0.0])[None, :, None], (S, 1, n)) + 0.01 * np.sin(st["imu_time"])[:, None, :]
    quat /= np.linalg.norm(quat, axis=1, keepdims=True)
    d = _dev(st)
    prm = est_mod.robot_params("go1")
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
    P_dev = mhe.mhe_qp_.P_window()
    assert P_dev.shape == (20, 9, 9, n)
    h = mhe._hd
    P_raw = torch.empty(20, 81, n, dtype=torch.float64, device="cuda")
    K = C.c_int32()
    h.check(h.L.dekf_get_window_cov(h.h, C.c_void_p(P_raw.data_ptr()), C.byref(K)), "dekf_get_window_cov")
    assert K.value == 20 and torch.equal(P_raw.view(20, 9, 9, n), P_dev)
    host = np.zeros((20 * 81, n))
    h.check(h.L.dekf_get_host(h.h, 10, host.ctypes.data_as(C.c_void_p)), "dekf_get_host")
    assert np.array_equal(host.reshape(20, 9, 9, n), P_dev.cpu().numpy())
    # the batched class over the same stream without the host-side orientations: its own window_cov() and the device getter
    be = _est(est_mod, n)
    for s in range(S):
        be.step(s, est_mod.robot_store.from_stream(d, s))
    hb = be._hd
    h.check(hb.L.dekf_get_window_cov(hb.h, C.c_void_p(P_raw.data_ptr()), None), "dekf_get_window_cov")
    assert torch.equal(be.window_cov(), P_raw.view(20, 9, 9, n))
    # C++ facade over the same stream and orientations
    so = build.build()
    src, exe = tmp_path / "cov_main.cpp", str(tmp_path / "cov_main")
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
    P_cpp = np.fromfile(outp, np.float64)
    assert P_cpp.size == 20 * 81 * n and np.array_equal(P_cpp.reshape(20, 9, 9, n), P_dev.cpu().numpy())
