"""Smoothed MHE window (dekf_get_window): every state block of MHEproblem::solution (MheSrb.hpp:58-112), computed by a
backward (Rauch-Tung-Striebel) pass over the filtered states of the window (csrc/estimator_core.cuh, mhe_window_smooth).

CPU: the kernel body compiled for the host (tests/hostsim) against the oracle's exact primal (Mhe.solution(), pinned to the
compiled reference's `solution`), per tick, every window state.  GPU (-m gpu): the device getter against the oracle and the
host build, its consistency with the step outputs, the pipelined run, the error paths and the three host-side mirrors."""
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
TOL_V64, TOL_REL64, TOL_V32 = 1e-6, 1e-7, 1e-4


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
    out = {"ragged_n20": (synth.to_numpy(synth.make_stream(16, 200, vo_jitter=True)), 20, 200)}
    for name in ("mhe_n5", "mhe_n5_late"):
        out[name] = _golden(name)
    return out


def oracle_windows(oracle, st, N, rate, inst):
    """The oracle's live Mhe, stepped like the reference: after every update(T) the state blocks of solution(), [S][N][9][len(inst)]
    (rows K = min(T+1, N) and beyond NaN)."""
    S = st["gyro"].shape[0]
    W = np.full((S, N, 9, len(inst)), np.nan)
    prm = oracle.go1_params(N=N)
    for j, i in enumerate(inst):
        ekf = oracle.Ekf(oracle.ekf_params(rate=rate))
        m = oracle.Mhe(prm)
        for s in range(S):
            vo = vq = None
            if st["vo_flag"][s, i]:
                vo = (st["vo_time_pre"][s, i], st["vo_time_now"][s, i], st["vo_rel_p"][s, :, i])
                vq = st["vo_quat"][s, :, i]
            ekf.tick(st["gyro"][s, :, i], st["accel"][s, :, i], st["imu_time"][s, i], vq, st["vo_time_now"][s, i])
            q, _ = ekf.get()
            m.step(s, imu_time=st["imu_time"][s, i], accel=st["accel"][s, :, i], gyro=st["gyro"][s, :, i], quat=q,
                   joint_pos=st["joint_pos"][s, :, i], joint_vel=st["joint_vel"][s, :, i], foot_force=st["foot_force"][s, :, i],
                   vo=vo)
            if s < 1:
                continue
            ds, dm, dc, _, _ = m.dims()
            sol, K, stride = m.solution(), min(s + 1, N), 2 * ds + dm + dc   # var_x(j) = j (2 ds + dm + dc), oracle/mhe.c
            W[s, :K, :, j] = np.array([sol[k * stride:k * stride + 9] for k in range(K)])
    return W


def window_errors(W, Wo):
    """(max velocity error, max over windows of component error / max(1, |x|max of the window))."""
    S = W.shape[0]
    dv, rel = 0.0, 0.0
    for s in range(1, S):
        K = min(s + 1, W.shape[1])
        d = np.abs(W[s, :K] - Wo[s, :K])
        assert np.isfinite(d).all()
        dv = max(dv, d[:, 3:6].max())
        scale = np.maximum(1.0, np.abs(Wo[s, :K]).max(axis=(0, 1)))
        rel = max(rel, (d.max(axis=(0, 1)) / scale).max())
    return dv, rel


@pytest.fixture(scope="module")
def cases(oracle):
    out = {}
    for name, (st, N, rate) in _streams().items():
        n = st["gyro"].shape[2]
        out[name] = (st, N, rate, oracle_windows(oracle, st, N, rate, list(range(n))))
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["ragged_n20", "mhe_n5", "mhe_n5_late"])
@pytest.mark.parametrize("precision", [0, 1])
def test_host_window_matches_oracle(cases, name, precision):
    """Every window state of every tick, both solve modes: fp64 velocity <= 1e-6 m/s and every component <= 1e-7 max(1, |x|max);
    fp32 velocity <= 1e-4 m/s."""
    import pywindowsim as ws
    st, N, rate, Wo = cases[name]
    for mode in (0, 1):
        r = ws.run(st, _hs_cfg(N=N, ekf_rate=rate, window_solve=mode, precision=precision))
        dv, rel = window_errors(r["window"], Wo)
        print(f"{name} precision={precision} mode={mode}: max |dv| {dv:.3e} m/s, max rel {rel:.3e}")
        if precision == 0:
            assert dv < TOL_V64 and rel < TOL_REL64
        else:
            assert dv < TOL_V32


@pytest.mark.parametrize("precision", [0, 1])
def test_host_window_last_row_and_modes_bit_identical(precision):
    """Row K-1 is the step's x bit for bit; the FULL-mode window (forward sweep from the arrival cost into a scratch ring)
    equals the INCREMENTAL-mode window (checkpoint ring) bit for bit."""
    import pywindowsim as ws
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(8, 160, vo_jitter=True))
    a = ws.run(st, _hs_cfg(window_solve=0, precision=precision))
    b = ws.run(st, _hs_cfg(window_solve=1, precision=precision))
    Wa, Wb = a["window"], b["window"]
    assert np.array_equal(np.isnan(Wa), np.isnan(Wb)) and np.array_equal(Wa[~np.isnan(Wa)], Wb[~np.isnan(Wb)])
    for s in range(1, Wa.shape[0]):
        K = min(s + 1, Wa.shape[1])
        assert np.array_equal(Wa[s, K - 1], a["x"][s]) and np.array_equal(Wb[s, K - 1], b["x"][s])
        assert np.isnan(Wa[s, K:]).all()


def _tally(name):
    src = os.path.join(HERE, "hostsim", name + ".cpp")
    out = os.path.join(HERE, "hostsim", "_build", name)
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", out, src])
    return json.loads(subprocess.check_output([out]).decode())


def test_probe_flop_constants_match_tally():
    tally = _tally("window_flopcount")
    tick = _tally("flopcount")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import window_probe
    for k in ("window_back", "window_back_vo", "window_fwd", "window_fwd_vo"):
        assert window_probe.FLOPS[k] == tally[k], (k, window_probe.FLOPS[k], tally[k])
    # the FULL-mode forward stage is the tick's incremental-sweep stage (leg rows + time update, P_pp carried)
    assert window_probe.FLOPS["window_fwd"] == tick["meas_update_pp"] + tick["propagate_pp"]
    assert window_probe.FLOPS["window_fwd_vo"] == tick["meas_update_pp"] + tick["propagate_vo_pp"]


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
def test_device_window_matches_oracle(est_mod, oracle, n, precision):
    """Getter every tick for 200 ticks; 32 instances against the oracle; last row == x and FULL == INCREMENTAL bit for bit."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, N, sel = 200, 20, np.linspace(0, n - 1, 32).astype(int)
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    st = synth.to_numpy({k: v[..., torch.as_tensor(sel, device="cuda")] for k, v in d.items()})
    Wo = oracle_windows(oracle, st, N, 200, list(range(len(sel))))
    full, incr = _est(est_mod, n, precision, 0), _est(est_mod, n, precision, 1)
    W = np.full((S, N, 9, len(sel)), np.nan)
    idx = torch.as_tensor(sel, device="cuda")
    for s in range(S):
        store = est_mod.robot_store.from_stream(d, s)
        full.step(s, store)
        incr.step(s, store)
        if s < 1:
            continue
        wf, wi = full.window(), incr.window()
        assert wf.shape == (min(s + 1, N), 9, n)
        assert torch.equal(wf, wi)
        assert torch.equal(wf[-1], full.x_MHE_) and torch.equal(wi[-1], incr.x_MHE_)
        W[s, :wf.shape[0]] = wf[..., idx].cpu().numpy()
    dv, rel = window_errors(W, Wo)
    print(f"n={n} {precision}: max |dv| {dv:.3e} m/s, max rel {rel:.3e}")
    if precision == "fp64":
        assert dv < TOL_V64 and rel < TOL_REL64
    else:
        assert dv < TOL_V32


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("mode", [0, 1])
def test_device_window_agrees_with_host_build(est_mod, precision, mode):
    """Device getter against the host build of the same kernel body, 64 instances x 160 ticks.  The two do not see bit-identical
    filtered states: the stage records come from the kinematics, whose sin / cos round differently on the device and in the
    host's libm, so x_T itself differs in the last bits.  The window may differ from the host build's by no more than a small
    multiple of that, relative to the window's scale."""
    import pywindowsim as ws
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(64, 160, vo_jitter=True))
    r = ws.run(st, _hs_cfg(window_solve=mode, precision=precision))
    est = _est(est_mod, 64, ("fp64", "fp32")[precision], mode)
    d = _dev(st)
    dx, dw = 0.0, 0.0
    for s in range(160):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        if s >= 1:
            w = est.window().cpu().numpy()
            wh = r["window"][s, :w.shape[0]]
            scale = max(1.0, np.abs(wh).max())
            dx = max(dx, np.abs(est.x_MHE_.cpu().numpy() - r["x"][s]).max() / scale)
            dw = max(dw, np.abs(w - wh).max() / scale)
    print(f"precision={precision} mode={mode}: device vs host build, x_T {dx:.3e}, window {dw:.3e} (relative)")
    assert dw <= (1e-12 if precision == 0 else 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [20000, 65536])
@pytest.mark.parametrize("mode", [0, 1])
def test_run_then_window_equals_single_steps(est_mod, n, mode):
    """dekf_run (pipelined, internal streams joined into the handle's stream) followed by the getter == single steps + getter."""
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S = 150
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    vo = [bool(d["vo_flag"][s].any()) for s in range(S)]
    a, b = _est(est_mod, n, "fp64", mode), _est(est_mod, n, "fp64", mode)
    a.run(0, S, d, vo)
    wa = a.window()
    for s in range(S):
        b.step(s, est_mod.robot_store.from_stream(d, s))
    wb = b.window()
    assert wa.shape == (20, 9, n) and torch.equal(wa, wb)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_getter_changes_no_output(est_mod, mode):
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 120, 512
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")
    a, b = _est(est_mod, n, "fp64", mode), _est(est_mod, n, "fp64", mode)
    for s in range(S):
        store = est_mod.robot_store.from_stream(d, s)
        a.step(s, store)
        b.step(s, store)
        if s >= 1:
            a.window()
        for k in ("quaternion_", "x_MHE_", "v_MHE_b_", "contact_", "status_"):
            ta, tb = getattr(a, k), getattr(b, k)
            if ta.is_floating_point():  # x / v_body are NaN before the first update
                assert torch.equal(ta.isnan(), tb.isnan()) and torch.equal(ta.nan_to_num(), tb.nan_to_num()), (s, k)
            else:
                assert torch.equal(ta, tb), (s, k)


@pytest.mark.gpu
def test_error_paths_and_reset(est_mod):
    import torch
    from decentralized_ekf_mhe_b200 import synth
    S, n = 60, 256
    d = synth.make_stream(n, S, vo_jitter=True, device="cuda")

    def rc_of(est, ptr=True):
        h = est._hd
        w = torch.empty(20, 9, n, dtype=torch.float64, device="cuda")
        rc = h.L.dekf_get_window(h.h, C.c_void_p(w.data_ptr()) if ptr else None, None)
        return rc, h.L.dekf_last_error(h.h).decode()

    for over in (dict(est_type=1), dict(leg_odom_type=1), dict(v_box_enable=1, v_box_lo=(-1, -1, -1), v_box_hi=(1, 1, 1)),
                 dict(x_box_mask=1 << 3, x_box_lo=(0, 0, 0, -1, 0, 0, 0, 0, 0), x_box_hi=(0, 0, 0, 1, 0, 0, 0, 0, 0))):
        e = _est(est_mod, n, **over)
        for s in range(3):
            e.step(s, est_mod.robot_store.from_stream(d, s))
        rc, msg = rc_of(e)
        assert rc == -1 and msg.startswith("dekf_get_window"), (over, rc, msg)
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
        assert rc_of(e, ptr=False)[0] == -1            # null x
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
        assert torch.equal(e.window(), fresh.window())


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
  const std::vector<double> w = mhe.mhe_qp_.x_window();
  std::FILE *o = std::fopen(argv[2], "wb");
  std::fwrite(w.data(), sizeof(double), w.size(), o);
  std::fclose(o);
  return 0;
}
"""


@pytest.mark.gpu
def test_host_getter_python_class_api_and_cpp_facade_equal_device(est_mod, tmp_path):
    """dekf_get_host(DEKF_GET_WINDOW_X), DecentralizedEstimation.mhe_qp_.x_window() and the C++ facade's mhe_qp_.x_window()
    all return the device getter's window."""
    import torch
    from decentralized_ekf_mhe_b200 import build, synth
    n, S = 48, 90
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
    w_dev = mhe.mhe_qp_.x_window()
    assert w_dev.shape == (20, 9, n)
    h = mhe._hd
    host = np.zeros((20 * 9, n))
    h.check(h.L.dekf_get_host(h.h, 9, host.ctypes.data_as(C.c_void_p)), "dekf_get_host")
    assert np.array_equal(host.reshape(20, 9, n), w_dev.cpu().numpy())
    # C++ facade over the same stream and orientations
    so = build.build()
    src, exe = tmp_path / "window_main.cpp", str(tmp_path / "window_main")
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
    w_cpp = np.fromfile(outp, np.float64)
    assert w_cpp.size == 20 * 9 * n and np.array_equal(w_cpp.reshape(20, 9, n), w_dev.cpu().numpy())


@pytest.mark.gpu
def test_smoothed_lagged_velocity_beats_filtered(est_mod):
    """Velocity of stage T-10 against the ground truth: the smoothed estimate (window row K-11 at tick T) against the filtered
    one (x of tick T-10), pooled over all instances and ticks T >= N."""
    from decentralized_ekf_mhe_b200 import synth
    S, n, N, lag = 200, 256, 20, 10
    d = synth.make_stream(n, S, vo_jitter=True, truth=True, device="cuda")
    vt = d["v_true"].cpu().numpy()
    est = _est(est_mod, n)
    xs, es, ef = [], [], []
    for s in range(S):
        est.step(s, est_mod.robot_store.from_stream(d, s))
        xs.append(est.x_MHE_.cpu().numpy())
        if s >= N:
            w = est.window().cpu().numpy()
            es.append(w[N - 1 - lag, 3:6] - vt[s - lag])
            ef.append(xs[s - lag][3:6] - vt[s - lag])
    rs, rf = np.sqrt(np.mean(np.square(es))), np.sqrt(np.mean(np.square(ef)))
    print(f"lag-{lag} velocity RMS error: smoothed {rs:.5f} m/s, filtered {rf:.5f} m/s")
    assert rs < rf
