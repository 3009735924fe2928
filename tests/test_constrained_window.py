"""Window of a state-constrained handle (dekf_get_constrained_window): the optimum of every window state, its covariance with the
active bounds as equalities and the active set, read from the scratch of the last active-set solve (csrc/box_window.cuh).

Handles: the velocity box (PogoX, BASELINE config 4), general component bounds (x_box_mask) and general linear rows
(dekf_add_state_rows).  Oracle: the oracle's window QP of the same tick -- Mhe.solution() for the mean, and for the covariance
the KKT matrix of Mhe.export_qp() with its equality rows plus one row per bound the getter reports active, solved for the unit
columns of the state variables.  CPU: the header code in the host build (tests/hostsim/box_window_hostsim.cpp).  GPU (-m gpu):
the device getter against the oracle and the host build, both scratch layouts, the pipelined run, output invariance, the
error paths and the mirrors."""
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

POGOX = dict(robot=2, num_legs=1, contact_effort_threshold=100.0, p_ib=(0.0, 0.0, 0.0), p_imu_2_opti=(0.0, 0.0, 0.0))
BOX_LO, BOX_HI = (-0.45, -0.03, -0.015), (0.55, 0.03, 0.015)
MASK = (1 << 3) | (1 << 2) | (7 << 6)
LO9 = (0, 0, -2e-4, 0.47, 0, 0, -0.004, -0.004, -0.004)
HI9 = (0, 0, 2e-4, 0.52, 0, 0, 0.004, 0.004, 0.004)
TICKS = (1, 4, 12, 19, 20, 21, 33, 47)   # below, at and above N = 20


def _rows3():
    A = np.zeros((3, 9))
    A[0, 3], A[0, 5] = 1.0, 0.5          # v_x + 0.5 v_z
    A[1, 6], A[1, 7] = 1.0, -1.0         # b_x - b_y
    A[2, 2], A[2, 8] = 1.0, 0.02         # p_z + 0.02 b_z
    return A, np.array([0.47, -0.003, -2e-4]), np.array([0.52, 0.003, 2e-4])


def _kind(name):
    """(config overrides, oracle overrides, rows for the host build / the handle, bounded rows R [m][9], lo [m], hi [m]) of a
    handle kind; rows in the public order of the active words."""
    if name == "vbox":
        R = np.eye(9)
        lo, hi = np.full(9, -np.inf), np.full(9, np.inf)
        lo[3:6], hi[3:6] = BOX_LO, BOX_HI
        kw = dict(v_box_enable=1, v_box_lo=BOX_LO, v_box_hi=BOX_HI)
        return kw, kw, None, R, lo, hi
    if name == "xbox":
        R = np.eye(9)
        lo = np.where([(MASK >> a) & 1 for a in range(9)], LO9, -np.inf)
        hi = np.where([(MASK >> a) & 1 for a in range(9)], HI9, np.inf)
        kw = dict(x_box_mask=MASK, x_box_lo=LO9, x_box_hi=HI9)
        return kw, kw, None, R, lo, hi
    A3, lo3, hi3 = _rows3()
    xlo, xhi = [0.0] * 9, [0.0] * 9
    xlo[4], xhi[4] = -0.02, 0.02
    kw = dict(x_box_mask=1 << 4, x_box_lo=tuple(xlo), x_box_hi=tuple(xhi))
    okw = dict(kw, x_row_count=3, x_row_a=tuple(A3.reshape(-1)) + (0.0,) * 54, x_row_lo=tuple(lo3) + (0.0,) * 6,
               x_row_hi=tuple(hi3) + (0.0,) * 6)
    R = np.vstack([A3, np.eye(9)[4:5]])
    return kw, okw, (A3, lo3, hi3), R, np.concatenate([lo3, [-0.02]]), np.concatenate([hi3, [0.02]])


def _hs_cfg(go1=False, **over):
    import pyhostsim as hs
    from decentralized_ekf_mhe_b200.params import DekfConfig
    lib = C.CDLL(hs.build())
    cfg = DekfConfig()
    lib.hostsim_default_go1(C.byref(cfg))
    cfg.ekf_rate = 200
    if not go1:
        cfg.update(**POGOX)
    cfg.update(**over)
    return cfg


def _stream(n=3, S=48):
    from decentralized_ekf_mhe_b200 import synth
    return synth.to_numpy(synth.make_stream(n, S, robot="pogox", vo_jitter=True))


def oracle_window(oracle, st, okw, R, lo, hi, act_of, inst, ticks):
    """{T: dict(x [K][9][n], P [K][9][9][n], mult [K][2m][n])} from the oracle's window QP of tick T.  act_of(T, i): [K] active
    words (public encoding) whose bounds join the KKT rows; mult: the oracle's multiplier of every bound at ITS optimum (lower
    bounds in 0..m-1, upper in m..2m-1; 0 where the bound is not at the optimum)."""
    m = R.shape[0]
    out = {}
    prm = oracle.go1_params(**POGOX, **okw)
    for j, i in enumerate(inst):
        ekf = oracle.Ekf(oracle.ekf_params(rate=200))
        mh = oracle.Mhe(prm)
        for s in range(max(ticks) + 1):
            vo = vq = None
            if st["vo_flag"][s, i]:
                vo = (st["vo_time_pre"][s, i], st["vo_time_now"][s, i], st["vo_rel_p"][s, :, i])
                vq = st["vo_quat"][s, :, i]
            ekf.tick(st["gyro"][s, :, i], st["accel"][s, :, i], st["imu_time"][s, i], vq, st["vo_time_now"][s, i])
            q, _ = ekf.get()
            mh.step(s, imu_time=st["imu_time"][s, i], accel=st["accel"][s, :, i], gyro=st["gyro"][s, :, i], quat=q,
                    joint_pos=st["joint_pos"][s, :, i], joint_vel=st["joint_vel"][s, :, i],
                    foot_force=st["foot_force"][s, :, i], vo=vo)
            if s not in ticks:
                continue
            ds, dm, dc, nV, _ = mh.dims()
            H, g, A, l, u = mh.export_qp()
            z = mh.solution()
            K, stride = min(s + 1, 20), 2 * ds + dm + dc
            xi = [k * stride for k in range(K)]
            o = out.setdefault(s, dict(x=np.zeros((K, 9, len(inst))), P=np.zeros((K, 9, 9, len(inst))),
                                       mult=np.zeros((K, 2 * m, len(inst)))))
            o["x"][:, :, j] = np.array([z[p:p + 9] for p in xi])
            eq = np.abs(u - l) < 1e-9
            Ae = A[eq]
            # the oracle's own multipliers (bounds at its optimum)
            val = o["x"][:, :, j] @ R.T
            at = []
            for k in range(K):
                for r in range(m):
                    if abs(val[k, r] - hi[r]) < 1e-9 * max(1.0, abs(hi[r])):
                        at.append((k, r, 1))
                    elif abs(val[k, r] - lo[r]) < 1e-9 * max(1.0, abs(lo[r])):
                        at.append((k, r, 0))
            B = np.zeros((len(at), nV))
            for q_, (k, r, _) in enumerate(at):
                B[q_, xi[k]:xi[k] + 9] = R[r]
            G = np.vstack([Ae, B]).T
            sol, *_ = np.linalg.lstsq(G, -(H @ z + g), rcond=None)
            for (k, r, up), w in zip(at, sol[Ae.shape[0]:]):
                o["mult"][k, r + m * up, j] = w
            # covariance with the bounds the getter reports active
            words = act_of(s, i)
            rows = [(k, r) for k in range(K) for r in range(m) if (int(words[k]) >> r | int(words[k]) >> (9 + r)) & 1]
            Bc = np.zeros((len(rows), nV))
            for q_, (k, r) in enumerate(rows):
                Bc[q_, xi[k]:xi[k] + 9] = R[r]
            Cm = np.vstack([Ae, Bc])
            nc = Cm.shape[0]
            KKT = np.block([[H, Cm.T], [Cm, np.zeros((nc, nc))]])
            idx = np.concatenate([np.arange(p, p + 9) for p in xi])
            E = np.zeros((KKT.shape[0], len(idx)))
            E[idx, np.arange(len(idx))] = 1.0
            X = np.linalg.solve(KKT, E)[idx]
            for k in range(K):
                o["P"][k, :, :, j] = X[9 * k:9 * k + 9, 9 * k:9 * k + 9]
    return out


def cov_error(P, Po):
    """max correlation-scaled error of P [K][9][9][n] against Po over the free coordinates: those whose oracle variance is not
    negligible against the largest of its block (a coordinate fixed by an active bound has variance zero up to round-off)."""
    d = np.sqrt(np.abs(np.einsum("kiin->kin", Po)))
    free = d > 1e-6 * d.max(axis=1, keepdims=True)
    s = d[:, :, None, :] * d[:, None, :, :]
    ok = free[:, :, None, :] & free[:, None, :, :]
    return float((np.abs(P - Po)[ok] / s[ok]).max())


@pytest.fixture(scope="module")
def host_cases(oracle):
    """{kind: (stream, host result, oracle result at TICKS)} for the three handle kinds, fp64."""
    import pyboxwindowsim as bw
    out = {}
    st = _stream()
    for name in ("vbox", "xbox", "rows"):
        kw, okw, rows, R, lo, hi = _kind(name)
        r = bw.run_window(st, _hs_cfg(**kw), rows=rows)
        o = oracle_window(oracle, st, okw, R, lo, hi, lambda T, i: r["act"][T, :min(T + 1, 20), i], list(range(st["gyro"].shape[2])), TICKS)
        out[name] = (st, r, o, R, lo, hi)
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_host_mean_matches_oracle(host_cases, name):
    """x within 1e-8 of the state blocks of Mhe.solution() at ticks below, at and above N; row K-1 is the step's x_T bit for bit."""
    st, r, o, *_ = host_cases[name]
    err = 0.0
    for T, ot in o.items():
        K = ot["x"].shape[0]
        err = max(err, float(np.abs(r["win"][T, :K] - ot["x"]).max()))
        assert np.array_equal(r["win"][T, K - 1], r["x"][T])
    for T in range(1, r["x"].shape[0]):
        assert np.array_equal(r["win"][T, min(T + 1, 20) - 1], r["x"][T])
    print(f"{name}: max |x - oracle| {err:.3e}")
    assert err < 1e-8


@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_host_cov_matches_dense_kkt(host_cases, name):
    """P against the dense KKT inverse with the equality rows plus the reported active bounds, correlation-scaled, 1e-9;
    fixed components exactly zero."""
    st, r, o, R, lo, hi = host_cases[name]
    err, nact = 0.0, 0
    for T, ot in o.items():
        K = ot["P"].shape[0]
        P = r["cov"][T, :K]
        err = max(err, cov_error(P, ot["P"]))
        act = r["act"][T, :K]
        nact += int((act != 0).sum())
        if name != "rows":
            fx = (act | (act >> 9)) & 0x1ff
            for a in range(9):
                sel = ((fx >> a) & 1).astype(bool)
                assert (P[:, a, :, :].transpose(0, 2, 1)[sel] == 0).all() and (P[:, :, a, :].transpose(0, 2, 1)[sel] == 0).all()
    print(f"{name}: max correlation-scaled error {err:.3e}, {nact} active words")
    assert nact > 0
    assert err < 1e-9


@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_host_active_set_matches_oracle(host_cases, name):
    """Every bound whose oracle multiplier is clearly nonzero is reported active, and every reported bound is at its value."""
    st, r, o, R, lo, hi = host_cases[name]
    m = R.shape[0]
    seen = 0
    for T, ot in o.items():
        K = ot["x"].shape[0]
        act = r["act"][T, :K].astype(np.int64)
        mult = ot["mult"]
        scale = np.abs(mult).max() + 1e-300
        for side in (0, 1):
            for rr in range(m):
                bit = (act >> (rr + 9 * side)) & 1
                clear = np.abs(mult[:, rr + m * side]) > 1e-6 * scale
                seen += int(clear.sum())
                assert (bit[clear] == 1).all(), (T, rr, side)
                val = np.einsum("c,kcn->kn", R[rr], r["win"][T, :K])
                bound = hi[rr] if side else lo[rr]
                assert (np.abs(val[bit == 1] - bound) <= 1e-9 * max(1.0, abs(bound))).all()
    assert seen > 0


@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_host_invariants(host_cases, name):
    """Every block exactly symmetric; the free sub-block positive definite; on rows handles a_i P a_i' ~ 0 for active rows."""
    st, r, o, R, lo, hi = host_cases[name]
    S, n = r["x"].shape[0], r["x"].shape[2]
    for T in range(1, S):
        K = min(T + 1, 20)
        P = r["cov"][T, :K]
        assert np.array_equal(P, P.transpose(0, 2, 1, 3))
        act = r["act"][T, :K]
        for k in range(K):
            for i in range(n):
                w = int(act[k, i])
                if name == "rows":
                    for rr in range(R.shape[0]):
                        if (w >> rr | w >> (9 + rr)) & 1:
                            a = R[rr]
                            assert abs(a @ P[k, :, :, i] @ a) <= 1e-12 * np.trace(P[k, :, :, i])
                    ev = np.linalg.eigvalsh(P[k, :, :, i])
                    assert ev.min() > -1e-12 * ev.max()
                else:
                    free = [a for a in range(9) if not ((w | (w >> 9)) >> a) & 1]
                    np.linalg.cholesky(P[k][np.ix_(free, free, [i])][:, :, 0])


def test_host_wide_bounds_equal_unconstrained_window():
    """Bounds that never bind: x and P equal the unconstrained window (window_hostsim, window_cov_hostsim) -- two independent
    algorithms for the same quantity."""
    import pyboxwindowsim as bw
    import pywindowcovsim as wc
    import pywindowsim as ws
    from decentralized_ekf_mhe_b200 import synth
    st = synth.to_numpy(synth.make_stream(4, 44, vo_jitter=True))   # Go1: the robot of the unconstrained harnesses
    r = bw.run_window(st, _hs_cfg(go1=True, v_box_enable=1, v_box_lo=(-50.0,) * 3, v_box_hi=(50.0,) * 3))
    assert (r["act"] == 0).all()
    u = ws.run(st, _hs_cfg(go1=True))
    c = wc.run_cov(st, _hs_cfg(go1=True))
    ex = ep = 0.0
    for T in range(1, st["gyro"].shape[0]):
        K = min(T + 1, 20)
        ex = max(ex, float(np.abs(r["win"][T, :K] - u["window"][T, :K]).max()))
        ep = max(ep, cov_error(r["cov"][T, :K], c["cov"][T, :K].reshape(K, 9, 9, -1)))
    print(f"wide bounds: x {ex:.3e}, P {ep:.3e}")
    assert ex < 1e-10 and ep < 1e-9


@pytest.mark.parametrize("name,cap", [("vbox", 2), ("xbox", 10)])
def test_host_capped_solve(name, cap):
    """A cap small enough to hit: row K-1 is x_T, P is NaN exactly on the capped instances, and on the general path the rows of
    an instance that reports the finite method's feasible iterate violate no bound."""
    import pyboxwindowsim as bw
    kw, _, rows, R, lo, hi = _kind(name)
    st = _stream(24, 40)
    r = bw.run_window(st, _hs_cfg(v_box_max_iter=cap, **kw), rows=rows)
    capped = r["capped"][1:] != 0
    assert capped.any()
    assert np.array_equal(capped, (r["status"][1:] & 64) != 0)
    feas = 0
    for T in range(1, st["gyro"].shape[0]):
        K = min(T + 1, 20)
        assert np.array_equal(r["win"][T, K - 1], r["x"][T])
        nanP = np.isnan(r["cov"][T, :K]).all(axis=(0, 1, 2))
        assert np.array_equal(nanP, r["capped"][T] != 0)
        assert not np.isnan(r["cov"][T, :K][..., ~nanP]).any()
        if name == "xbox":
            for i in np.nonzero(r["capped"][T] == 2)[0]:
                val = r["win"][T, :K, :, i] @ R.T
                assert (val <= hi + 1e-12).all() and (val >= lo - 1e-12).all()
                feas += 1
    if name == "xbox":
        assert feas > 0


def test_flop_tally_matches_probe():
    """tests/hostsim/box_window_flopcount.cpp (the header functions with a counting scalar) == the closed forms of the probe."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import window_probe as wp
    exe = os.path.join(HERE, "hostsim", "_build", "box_window_flopcount")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-o", exe,
                           os.path.join(HERE, "hostsim", "box_window_flopcount.cpp")])
    got = json.loads(subprocess.check_output([exe]).decode())
    assert got == wp.BOX_STAGE_FLOPS, (got, wp.BOX_STAGE_FLOPS)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _gpu():
    import torch as t
    from decentralized_ekf_mhe_b200 import estimator as E
    return t, E


def _device_run(name, n, S, precision="fp64", cap=0, rows_env=None, ticks_cb=None):
    """Step a PogoX handle of kind `name` S ticks; ticks_cb(s, est) after every step.  Returns (est, device stream)."""
    t, E = _gpu()
    from decentralized_ekf_mhe_b200 import synth
    kw, _, rows, *_ = _kind(name)
    if cap:
        kw = dict(kw, v_box_max_iter=cap)
    st_t = synth.make_stream(n, S, robot="pogox", vo_jitter=True, device="cuda")
    d = {k: v.contiguous() for k, v in st_t.items()}
    est = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200, **kw), n, precision=precision)
    if rows is not None:
        est.add_state_rows(*rows)
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
        if ticks_cb is not None:
            ticks_cb(s, est)
    return est, st_t


def _get(est):
    x, P, a = est.window(), est.window_cov(), est.window_active()
    return x.cpu().numpy(), P.cpu().numpy(), a.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("n", [300, 301])   # 301: the last warp of the team layout holds one instance
@pytest.mark.parametrize("name", ["vbox", "xbox", "rows"])
def test_device_matches_host_and_oracle(oracle, name, n, precision):
    """Device getter against the host build of the same ticks (the same header code) and the oracle, at the sampled ticks."""
    import pyboxwindowsim as bw
    t, E = _gpu()
    from decentralized_ekf_mhe_b200 import synth
    kw, okw, rows, R, lo_, hi_ = _kind(name)
    S = 34
    st_t = synth.make_stream(n, S, robot="pogox", vo_jitter=True)
    st = synth.to_numpy(st_t)
    d = {k: v.cuda().contiguous() for k, v in st_t.items()}
    est = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200, **kw), n, precision=precision)
    if rows is not None:
        est.add_state_rows(*rows)
    got = {}
    for s in range(S):
        est.step(s, E.robot_store.from_stream(d, s))
        if s in (1, 12, 20, 33):
            x, P, a = _get(est)
            got[s] = (x, P, a, est.x_MHE_.cpu().numpy())
    est.close()
    m = 6
    sub = {k: np.ascontiguousarray(v[..., :m]) for k, v in st.items()}
    hres = bw.run_window(sub, _hs_cfg(precision=0 if precision == "fp64" else 1, **kw), rows=rows)
    o = oracle_window(oracle, sub, okw, R, lo_, hi_, lambda T, i: got[T][2][:, i], list(range(m)), tuple(got))
    tol_x, tol_p = (1e-8, 1e-8) if precision == "fp64" else (1e-4, 1e-3)
    ex = ep = eh = 0.0
    for T, (x, P, a, xT) in got.items():
        K = min(T + 1, 20)
        assert x.shape == (K, 9, n) and P.shape == (K, 9, 9, n) and a.shape == (K, n)
        assert np.array_equal(x[K - 1], xT)
        assert np.array_equal(P, P.transpose(0, 2, 1, 3)) and np.isfinite(P).all()
        ex = max(ex, float(np.abs(x[:, :, :m] - o[T]["x"]).max()))
        ep = max(ep, cov_error(P[..., :m], o[T]["P"]))
        if precision == "fp64":
            eh = max(eh, float(np.abs(x[:, :, :m] - hres["win"][T, :K]).max()))
    print(f"{name} n={n} {precision}: x vs oracle {ex:.3e}, P vs oracle {ep:.3e}, x vs host {eh:.3e}")
    assert ex < tol_x and ep < tol_p and eh < 1e-9


@pytest.mark.gpu
def test_team_layout_equals_serial_layout(monkeypatch):
    """The velocity box through the team solve (default) and the serial solve (DEKF_BOX_SERIAL=1) give the same window."""
    res = []
    for serial in ("0", "1"):
        monkeypatch.setenv("DEKF_BOX_SERIAL", serial)
        est, _ = _device_run("vbox", 3001, 30)
        res.append(_get(est))
        est.close()
    (xa, Pa, aa), (xb, Pb, ab) = res
    assert np.abs(xa - xb).max() < 1e-6
    assert cov_error(Pa, Pb) < 1e-6
    assert (aa != ab).mean() < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("name,cap", [("vbox", 0), ("xbox", 0), ("rows", 0), ("vbox", 2), ("xbox", 10)])
def test_xT_identity_and_no_side_effects(name, cap):
    """Row K-1 equals dekf_outputs.x bit for bit on every tick; calling the getter between ticks changes no step output; capped
    instances have all-NaN P blocks and finite x."""
    t, E = _gpu()
    outs = []
    for call in (False, True):
        xs = []

        def cb(s, est):
            if s >= 1 and call:
                x, P, a = est.window(), est.window_cov(), est.window_active()
                K = x.shape[0]
                assert t.equal(x[K - 1], est.x_MHE_)
                capped = (est.status_ & 64) != 0
                assert t.isnan(P[..., capped]).all() and not t.isnan(P[..., ~capped]).any()
            xs.append((est.x_MHE_.clone(), est.v_MHE_b_.clone(), est.status_.clone()))

        est, _ = _device_run(name, 400, 26, cap=cap, ticks_cb=cb)
        est.close()
        outs.append(xs)
    for s, ((a0, b0, c0), (a1, b1, c1)) in enumerate(zip(*outs)):
        assert t.equal(c0, c1)
        if s >= 1:   # tick 0 has no update: x and v_body are still NaN
            assert t.equal(a0, a1) and t.equal(b0, b1)


@pytest.mark.gpu
def test_run_equals_steps():
    """dekf_run followed by the getter equals single steps followed by the getter."""
    t, E = _gpu()
    from decentralized_ekf_mhe_b200 import synth
    n, S = 2000, 30
    kw = _kind("vbox")[0]
    st = synth.make_stream(n, S, robot="pogox", vo_jitter=True, device="cuda")
    d = {k: v.contiguous() for k, v in st.items()}
    vo = [bool(st["vo_flag"][s].any()) for s in range(S)]
    a = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200, **kw), n)
    a.run(0, S, d, vo)
    ra = _get(a)
    a.close()
    b = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200, **kw), n)
    for s in range(S):
        b.step(s, E.robot_store.from_stream(d, s))
    rb = _get(b)
    b.close()
    for u, v in zip(ra, rb):
        assert np.array_equal(u, v, equal_nan=True)


@pytest.mark.gpu
def test_wide_bounds_equal_unconstrained_getters():
    """Wide bounds on the device equal dekf_get_window / dekf_get_window_cov of an unconstrained fp64 handle."""
    t, E = _gpu()
    from decentralized_ekf_mhe_b200 import synth
    n, S = 500, 30
    st = synth.make_stream(n, S, robot="pogox", vo_jitter=True, device="cuda")
    d = {k: v.contiguous() for k, v in st.items()}
    a = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200, v_box_enable=1, v_box_lo=(-50.0,) * 3, v_box_hi=(50.0,) * 3), n)
    b = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200), n)
    for s in range(S):
        a.step(s, E.robot_store.from_stream(d, s))
        b.step(s, E.robot_store.from_stream(d, s))
    xa, Pa, aa = _get(a)
    xb, Pb = b.window().cpu().numpy(), b.window_cov().cpu().numpy()
    a.close()
    b.close()
    assert (aa == 0).all()
    assert np.abs(xa - xb).max() < 1e-10
    assert cov_error(Pa, Pb) < 1e-9


@pytest.mark.gpu
def test_errors_and_reset():
    """All-null outputs and unconstrained handles: DEKF_EINVAL (the message names the getters to use); before the first
    update(T >= 1) and after dekf_reset: DEKF_ESTATE; the existing getters keep refusing constrained handles."""
    t, E = _gpu()
    from decentralized_ekf_mhe_b200 import _lib
    L = _lib.load()
    EINVAL, ESTATE = -1, -5   # include/dekf_b200.h
    est, _ = _device_run("vbox", 64, 1)
    h = est._hd
    K = C.c_int32()
    x = t.empty(20, 9, 64, dtype=t.float64, device="cuda")
    assert L.dekf_get_constrained_window(h.h, C.c_void_p(x.data_ptr()), None, None, C.byref(K)) == ESTATE
    est.close()
    est, st = _device_run("vbox", 64, 5)
    h = est._hd
    assert L.dekf_get_constrained_window(h.h, None, None, None, C.byref(K)) == EINVAL
    assert L.dekf_get_constrained_window(h.h, C.c_void_p(x.data_ptr()), None, None, C.byref(K)) == 0 and K.value == 5
    assert L.dekf_get_window(h.h, C.c_void_p(x.data_ptr()), C.byref(K)) == EINVAL
    assert L.dekf_reset(h.h) == 0
    assert L.dekf_get_constrained_window(h.h, C.c_void_p(x.data_ptr()), None, None, C.byref(K)) == ESTATE
    est.close()
    u = E.BatchedEstimator(E.robot_params("pogox", ekf_rate=200), 64)
    rc = L.dekf_get_constrained_window(u._hd.h, C.c_void_p(x.data_ptr()), None, None, C.byref(K))
    msg = L.dekf_last_error(u._hd.h).decode()
    u.close()
    assert rc == EINVAL and "dekf_get_window" in msg and "dekf_get_window_cov" in msg


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["vbox", "rows"])
def test_mirrors_equal_device_getter(name):
    """Host selectors 13-15 and the Python class API return what the device getter returns."""
    t, E = _gpu()
    from decentralized_ekf_mhe_b200 import _lib
    L = _lib.load()
    n = 128
    est, _ = _device_run(name, n, 24)
    h = est._hd
    x, P, a = _get(est)
    K = x.shape[0]
    hx = np.zeros(20 * 9 * n)
    hP = np.zeros(20 * 81 * n)
    ha = np.zeros(20 * n, np.uint32)
    for sel, buf in ((13, hx), (14, hP), (15, ha)):
        assert L.dekf_get_host(h.h, sel, buf.ctypes.data_as(C.c_void_p)) == 0
    assert np.array_equal(hx[:K * 9 * n].reshape(K, 9, n), x)
    assert np.array_equal(hP[:K * 81 * n].reshape(K, 9, 9, n), P)
    assert np.array_equal(ha[:K * n].reshape(K, n).astype(np.int64), a)
    est.close()
