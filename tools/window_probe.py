"""Cost of the smoothed-window getters (dekf_get_window, and dekf_get_window_cov in the cov_* fields) on a large batch;
with --foot, of dekf_get_foot_window on Go1 foot-state handles (x-only, P-only, x+P and one step, at each --foot-n); with --box,
of dekf_get_constrained_window on state-constrained handles (PogoX config 4 and Go1 with a velocity box on the team layout, general
rows on the serial layout); with --cross, of dekf_get_window_cross_cov against the covariance getter of each handle kind (P only,
C only, P + C on the same handle, alternated in the same process).

Go1, N = 20, 65,536 instances, fp64 and fp32 handles, ragged and lock-step VO arrival, both window_solve modes.  Per setup:
64 warm-up ticks (dekf_run), then the getter timed with CUDA events over --calls calls, then a tick with and without the
getter, alternated in the same process.  Algorithmic bytes come from the shapes, flops from the operation tally of
tests/hostsim/window_flopcount.cpp (FLOPS below; tests/test_window_smoother.py keeps them equal); the roofline denominators are
dekf_measure_copy_bw / dekf_measure_fma_peak of the same device, as in bench.py.  Writes one JSON file.

usage: python tools/window_probe.py --out profiles/window_probe_b200.json [--n 65536] [--calls 200] [--ticks 40]
       python tools/window_probe.py --foot --out profiles/foot_window_probe_b200.json [--foot-n 16384 65536] [--calls 20]
       python tools/window_probe.py --box --out profiles/box_window_probe_b200.json [--calls 50] [--ticks 20]
       python tools/window_probe.py --cross --out profiles/window_cross_probe_b200.json [--calls 20]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# operations per stage (add + mul + div + sqrt, an FMA counts 2): backward stage without / with a VO row (double arithmetic),
# FULL-mode forward stage (leg-odometry update + time update with P_pp, handle precision) without / with a VO row
FLOPS = {"window_back": 1165, "window_back_vo": 2331, "window_fwd": 1100, "window_fwd_vo": 1700}
# one backward stage of the covariance getter (dekf_get_window_cov, double arithmetic) without / with a VO row
# (tests/hostsim/window_cov_flopcount.cpp; tests/test_window_covariance.py keeps them equal)
FLOPS_COV = {"window_cov": 4786, "window_cov_vo": 6543}
# what the lag-one cross block of dekf_get_window_cross_cov adds per stage (double): the 9-state pass; the constrained pass and
# its V C V' on rows handles (tests/hostsim/window_cross_flopcount.cpp, with foot_stage_flops(L)["cross"]; kept equal by
# tests/test_window_cross_cov.py)
FLOPS_CROSS = {"window_cross": 1377, "box_cross": 2187, "box_rows_vcvt": 2916}


def algorithmic_bytes(N, K, esize, full):
    """Bytes per instance: filtered states (54 words) and the record fields the backward pass reads (16 words) for N stages,
    the double output; FULL mode adds the forward sweep's whole records (25 words) and the scratch-ring writes (54 words)."""
    b = N * (54 + 16) * esize + 72 * K
    if full:
        b += N * (25 + 54) * esize
    return b


def cov_algorithmic_bytes(N, K, esize, full):
    """Bytes per instance of dekf_get_window_cov: filtered covariances (45 words) and the record fields the backward pass reads
    (16 words) for N stages, the double output [K][81]; FULL mode adds the forward sweep as in algorithmic_bytes.  Re-reading
    P_{k+1}^s from the block just written is an L2 hit and not counted."""
    b = N * (45 + 16) * esize + 648 * K
    if full:
        b += N * (25 + 54) * esize
    return b


def cov_algorithmic_flops(K, n_vo, full):
    """(double flops, handle-precision flops) per instance of dekf_get_window_cov."""
    back = (K - 1 - n_vo) * FLOPS_COV["window_cov"] + n_vo * FLOPS_COV["window_cov_vo"]
    fwd = ((K - n_vo) * FLOPS["window_fwd"] + n_vo * FLOPS["window_fwd_vo"]) if full else 0
    return back, fwd


def algorithmic_flops(K, n_vo, full):
    """(double flops, handle-precision flops) per instance for a window of K stages with n_vo VO rows."""
    back = (K - 1 - n_vo) * FLOPS["window_back"] + n_vo * FLOPS["window_back_vo"]
    fwd = ((K - n_vo) * FLOPS["window_fwd"] + n_vo * FLOPS["window_fwd_vo"]) if full else 0
    return back, fwd



def foot_stage_flops(L):
    """Operations of the backward passes of dekf_get_foot_window per stage (double; tests/hostsim/foot_window_flopcount.cpp,
    tests/test_foot_window.py keeps them equal): mean x_k = L^-T (y - Y x_{k+1}); covariance P_k = L^-T (I + Y P Y') L^-1
    (ds columns of G, each P v, Y w and a back substitution, then ds back substitutions); cov_T = L_T^-T L_T^-1."""
    ds = 9 + 3 * L
    ny = 9 * ds + sum(ds - (9 + 3 * ((c - 9) // 3)) for c in range(9, ds))   # nonzeros of Y
    back = ds * ds
    # cross: the lag-one block C_k = -L^-T Y P_{k+1} of dekf_get_window_cross_cov, ds columns of Y (P e_c) and a back substitution
    return {"mean": 2 * ny + back, "cov": ds * (ds * (2 * ds - 1) + 2 * ny + back) + ds * back, "cov_T": 2 * ds * back,
            "cross": ds * (2 * ny - ds + back)}


def foot_words(L):
    """(stage record words W, nonzeros of L, nonzeros of Y) of the dekf_get_foot_window ring."""
    ds = 9 + 3 * L
    nl = ds * (ds + 1) // 2
    ny = 9 * ds + sum(ds - (9 + 3 * ((c - 9) // 3)) for c in range(9, ds))
    return nl + ny + ds, nl, ny


def foot_algorithmic(L, K, want_x, want_P):
    """(bytes, backward-pass double flops) per instance of one dekf_get_foot_window call over K states.  Bytes: the forward
    sweep's inputs (arrival cost, K leg records of 9L+1 words and K common records of 16 words), the ring written and read
    back ((K-1) W words each way), the outputs.  The forward sweep's flops (the step's own sweep, repeated) are not in the
    tally; the flop bound below is the backward passes only."""
    ds = 9 + 3 * L
    W, nl, _ = foot_words(L)
    words = nl + ds + K * (9 * L + 1 + 16) + 2 * (K - 1) * W + (K * ds if want_x else 0) + (K * ds * ds if want_P else 0)
    f = foot_stage_flops(L)
    flops = ((K - 1) * f["mean"] if want_x else 0) + (((K - 1) * f["cov"] + f["cov_T"]) if want_P else 0)
    return 8 * words, flops


def foot_main(a, torch, estimator, synth, peaks):
    """Go1 foot-state handles (leg_odom_type 1), N = 20, ragged VO, warm-up to K = N; x-only, P-only and x+P calls and one
    k_foot_team tick, per instance count."""
    N, warm, L = 20, 40, 4
    res = dict(card=card(), torch_device=torch.cuda.get_device_name(0), N=N, warmup_ticks=warm, calls=a.calls, peaks=peaks,
               foot_stage_flops=foot_stage_flops(L), ring_words_per_stage=foot_words(L)[0], runs=[])
    for n in a.foot_n:
        d = synth.make_stream(n, warm + 2 * a.ticks + 1, vo_jitter=True, device="cuda")
        vo = [bool(d["vo_flag"][s].any()) for s in range(d["gyro"].shape[0])]
        est = estimator.BatchedEstimator(estimator.robot_params("go1", ekf_rate=200, N=N, leg_odom_type=1), n, precision="fp64")
        est.run(0, warm, {k: v[:warm] for k, v in d.items()}, vo[:warm])
        h = est._hd
        ds = h.ds
        x = torch.empty(N, ds, n, dtype=torch.float64, device="cuda")
        P = torch.empty(N, ds * ds, n, dtype=torch.float64, device="cuda")
        K = torch.zeros(1, dtype=torch.int32)
        kp = C.cast(K.data_ptr(), C.POINTER(C.c_int32))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r = dict(n=n, T=warm - 1)
        for name, px, pP in (("x", x, None), ("P", None, P), ("xP", x, P)):
            call = lambda: h.check(h.L.dekf_get_foot_window(h.h, C.c_void_p(px.data_ptr()) if px is not None else None,
                                                            C.c_void_p(pP.data_ptr()) if pP is not None else None, kp),
                                   "dekf_get_foot_window")
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.calls):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.calls
            Kv = int(K.item())
            by, fl = foot_algorithmic(L, Kv, px is not None, pP is not None)
            t_bw = by * n / (peaks["copy_gbs"] * 1e9) * 1e3
            t_fl = fl * n / (peaks["fp64_tflops"] * 1e12) * 1e3
            r[name] = dict(K=Kv, ms_per_call=ms, bytes_per_instance=by, backward_double_flops_per_instance=fl, hbm_bound_ms=t_bw,
                           flop_bound_ms=t_fl, bound="hbm" if t_bw >= t_fl else "fma", roof_fraction=max(t_bw, t_fl) / ms)
        ticks = []
        for j in range(a.ticks):   # k_foot_team tick (the whole step) in the same process, for scale
            s = warm + j
            store = estimator.robot_store.from_stream(d, s)
            e0.record()
            est.step(s, store)
            e1.record()
            torch.cuda.synchronize()
            ticks.append(e0.elapsed_time(e1))
        r["tick_ms_median"] = sorted(ticks)[len(ticks) // 2]
        r["x_over_tick"] = r["x"]["ms_per_call"] / r["tick_ms_median"]
        r["device_bytes"] = est.device_bytes()
        print(json.dumps(r), flush=True)
        res["runs"].append(r)
        est.close()
        del est, x, P, d
        torch.cuda.empty_cache()
    res["card_after"] = card()
    return res

# covariance pass of dekf_get_constrained_window per stage (double): S_j = L^-T (I + F' S F) L^-1, S_{K-1} = L^-T L^-1, and
# P = V S V' on rows handles (tests/hostsim/box_window_flopcount.cpp; tests/test_constrained_window.py keeps them equal).  The
# mean x = V y of rows handles costs 9 x (9 mul + 9 add) = 162 per stage (box_row_V, double only: not in the tally).
BOX_STAGE_FLOPS = {"cov": 4374, "cov_T": 1458, "rows_vsvt": 2268}
BOX_MEAN_ROWS_FLOPS = 162


def box_algorithmic(K, want_x, want_P, rows, act_bytes):
    """(bytes, double flops) per instance of one dekf_get_constrained_window call over K states.  Bytes: the capped byte; x: the
    iterate (9 words) read and written per stage; P: the stage factor (L and F, 126 words) and the active word read, 81 words
    written per stage."""
    words = (18 * K if want_x else 0) + (207 * K if want_P else 0)
    by = 8 * words + 1 + (act_bytes * K if want_P else 0)
    fl = (BOX_MEAN_ROWS_FLOPS * K if (want_x and rows) else 0)
    if want_P:
        fl += (K - 1) * BOX_STAGE_FLOPS["cov"] + BOX_STAGE_FLOPS["cov_T"] + (K * BOX_STAGE_FLOPS["rows_vsvt"] if rows else 0)
    return by, fl


def box_main(a, torch, estimator, synth, peaks):
    """Constrained handles, N = 20, warm-up to K = N: x-only, P-only and x+P calls against the constrained tick's own time."""
    import numpy as np
    N, warm = 20, 40
    rows = np.zeros((3, 9))
    rows[0, 3], rows[0, 5] = 1.0, 0.5
    rows[1, 6], rows[1, 7] = 1.0, -1.0
    rows[2, 2], rows[2, 8] = 1.0, 0.02
    cases = [("pogox_vbox_team", "pogox", 16384, dict(v_box_enable=1, v_box_lo=(-0.45, -0.03, -0.015), v_box_hi=(0.55, 0.03, 0.015)), None),
             ("go1_vbox_team", "go1", 65536, dict(v_box_enable=1, v_box_lo=(-0.3, -0.1, -0.05), v_box_hi=(0.6, 0.1, 0.05)), None),
             ("pogox_rows_serial", "pogox", 16384, dict(x_box_mask=1 << 4, x_box_lo=(0.0, 0.0, 0.0, 0.0, -0.02, 0.0, 0.0, 0.0, 0.0),
                                                        x_box_hi=(0.0, 0.0, 0.0, 0.0, 0.02, 0.0, 0.0, 0.0, 0.0)),
              (rows, np.array([0.47, -0.003, -2e-4]), np.array([0.52, 0.003, 2e-4])))]
    res = dict(card=card(), torch_device=torch.cuda.get_device_name(0), N=N, warmup_ticks=warm, calls=a.calls, peaks=peaks,
               box_stage_flops=BOX_STAGE_FLOPS, box_mean_rows_flops=BOX_MEAN_ROWS_FLOPS, runs=[])
    for name, robot, n, kw, rws in cases:
        d = synth.make_stream(n, warm + a.ticks + 1, robot=robot, vo_jitter=True, device="cuda")
        est = estimator.BatchedEstimator(estimator.robot_params(robot, ekf_rate=200, N=N, **kw), n, precision="fp64")
        if rws is not None:
            est.add_state_rows(*rws)
        bind = []
        for s in range(warm):
            est.step(s, estimator.robot_store.from_stream(d, s))
            if s >= 1:
                bind.append(float((est.window_active()[-1] != 0).double().mean()))
        h = est._hd
        x = torch.empty(N, 9, n, dtype=torch.float64, device="cuda")
        P = torch.empty(N, 81, n, dtype=torch.float64, device="cuda")
        K = torch.zeros(1, dtype=torch.int32)
        kp = C.cast(K.data_ptr(), C.POINTER(C.c_int32))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r = dict(case=name, robot=robot, n=n, layout="team" if h.cfg.x_box_mask == 0 and rws is None else "serial", T=warm - 1,
                 steps_with_a_bound_active=float(np.mean([b > 0 for b in bind])), mean_fraction_of_instances_bound=float(np.mean(bind)))
        for cname, px, pP in (("x", x, None), ("P", None, P), ("xP", x, P)):
            call = lambda: h.check(h.L.dekf_get_constrained_window(h.h, C.c_void_p(px.data_ptr()) if px is not None else None,
                                                                   C.c_void_p(pP.data_ptr()) if pP is not None else None, None, kp),
                                   "dekf_get_constrained_window")
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.calls):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.calls
            Kv = int(K.item())
            by, fl = box_algorithmic(Kv, px is not None, pP is not None, rws is not None, 4 if h.cfg.x_box_mask or rws is not None else 1)
            t_bw = by * n / (peaks["copy_gbs"] * 1e9) * 1e3
            t_fl = fl * n / (peaks["fp64_tflops"] * 1e12) * 1e3
            r[cname] = dict(K=Kv, ms_per_call=ms, bytes_per_instance=by, double_flops_per_instance=fl, hbm_bound_ms=t_bw,
                            flop_bound_ms=t_fl, bound="hbm" if t_bw >= t_fl else "fma", roof_fraction=max(t_bw, t_fl) / ms)
        ticks = []
        for j in range(a.ticks):   # the constrained tick itself (the whole step), for scale
            s = warm + j
            store = estimator.robot_store.from_stream(d, s)
            e0.record()
            est.step(s, store)
            e1.record()
            torch.cuda.synchronize()
            ticks.append(e0.elapsed_time(e1))
        r["tick_ms_median"] = sorted(ticks)[len(ticks) // 2]
        r["xP_over_tick"] = r["xP"]["ms_per_call"] / r["tick_ms_median"]
        r["device_bytes"] = est.device_bytes()
        print(json.dumps(r), flush=True)
        res["runs"].append(r)
        est.close()
        del est, x, P, d
        torch.cuda.empty_cache()
    res["card_after"] = card()
    return res


def cross_main(a, torch, estimator, synth, peaks):
    """dekf_get_window_cross_cov against the P-only getter of each handle kind, N = 20, warm-up to K = N: P only (the kind's
    covariance getter), C only and P + C, alternated over --rounds rounds of --calls calls each (median per call reported).
    Bytes and flops: those of the P-only call plus the [K-1][ds*ds] output and the tally's cross flops; the C-only call of a
    9-state handle still writes its P blocks, to a two-block ring, and is counted as P + C."""
    N, warm = 20, 40
    vbox = dict(v_box_enable=1, v_box_lo=(-0.45, -0.03, -0.015), v_box_hi=(0.55, 0.03, 0.015))
    setups = [(f"go1_{p}_{'incr' if m else 'full'}", "go1", a.n, dict(window_solve=m), p) for p in ("fp64", "fp32") for m in (1, 0)]
    setups += [(f"go1_foot_{n}", "go1", n, dict(leg_odom_type=1), "fp64") for n in a.foot_n]
    setups += [("pogox_vbox_team", "pogox", 16384, vbox, "fp64"), ("go1_vbox", "go1", a.n, vbox, "fp64")]
    res = dict(card=card(), torch_device=torch.cuda.get_device_name(0), N=N, warmup_ticks=warm, calls=a.calls, rounds=a.rounds,
               peaks=peaks, cov_flops_per_stage=FLOPS_COV, cross_flops_per_stage=FLOPS_CROSS, foot_stage_flops=foot_stage_flops(4),
               box_stage_flops=BOX_STAGE_FLOPS,
               runs=[])
    for name, robot, n, kw, prec in setups:
        d = synth.make_stream(n, warm, robot=robot, vo_jitter=True, device="cuda")
        vo = [bool(d["vo_flag"][s].any()) for s in range(warm)]
        est = estimator.BatchedEstimator(estimator.robot_params(robot, ekf_rate=200, N=N, **kw), n, precision=prec)
        est.run(0, warm, d, vo)
        h = est._hd
        ds = h.ds
        P = torch.empty(N, ds * ds, n, dtype=torch.float64, device="cuda")
        Cc = torch.empty(N - 1, ds * ds, n, dtype=torch.float64, device="cuda")
        K = torch.zeros(1, dtype=torch.int32)
        kp = C.cast(K.data_ptr(), C.POINTER(C.c_int32))
        pp, cp = C.c_void_p(P.data_ptr()), C.c_void_p(Cc.data_ptr())
        if kw.get("v_box_enable"):
            p_only = lambda: h.check(h.L.dekf_get_constrained_window(h.h, None, pp, None, kp), "dekf_get_constrained_window")
        elif kw.get("leg_odom_type") == 1:
            p_only = lambda: h.check(h.L.dekf_get_foot_window(h.h, None, pp, kp), "dekf_get_foot_window")
        else:
            p_only = lambda: h.check(h.L.dekf_get_window_cov(h.h, pp, kp), "dekf_get_window_cov")
        calls = {"P": p_only,
                 "C": lambda: h.check(h.L.dekf_get_window_cross_cov(h.h, None, cp, kp), "dekf_get_window_cross_cov"),
                 "PC": lambda: h.check(h.L.dekf_get_window_cross_cov(h.h, pp, cp, kp), "dekf_get_window_cross_cov")}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = {k: [] for k in calls}
        for f in calls.values():
            for _ in range(3):
                f()
        torch.cuda.synchronize()
        for _ in range(a.rounds):
            for k, f in calls.items():
                e0.record()
                for _ in range(a.calls):
                    f()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.calls)
        Kv = int(K.item())
        if kw.get("v_box_enable"):
            by, fl = box_algorithmic(Kv, False, True, False, 4)
            fl_c = (Kv - 1) * FLOPS_CROSS["box_cross"]
        elif kw.get("leg_odom_type") == 1:
            by, fl = foot_algorithmic(4, Kv, False, True)
            fl_c = (Kv - 1) * foot_stage_flops(4)["cross"]
        else:
            cnt = torch.empty(n, dtype=torch.int32, device="cuda")
            h.check(h.L.dekf_get_window_vo_count(h.h, C.c_void_p(cnt.data_ptr())), "dekf_get_window_vo_count")
            n_vo = float(cnt.double().mean())
            full, esize = kw["window_solve"] == 0, 8 if prec == "fp64" else 4
            by = cov_algorithmic_bytes(N, Kv, esize, full)
            f64, fh = cov_algorithmic_flops(Kv, n_vo, full)
            fl = f64 + fh
            fl_c = (Kv - 1) * FLOPS_CROSS["window_cross"]
        r = dict(setup=name, robot=robot, n=n, precision=prec, ds=ds, K=Kv)
        for k in calls:
            b = by + (8 * (Kv - 1) * ds * ds if k != "P" else 0)
            f = fl + (fl_c if k != "P" else 0)
            ms = sorted(times[k])[len(times[k]) // 2]
            t_bw = b * n / (peaks["copy_gbs"] * 1e9) * 1e3
            t_fl = f * n / (peaks["fp64_tflops"] * 1e12) * 1e3
            r[k] = dict(ms_per_call=ms, ms_all_rounds=times[k], bytes_per_instance=b, flops_per_instance=f, hbm_bound_ms=t_bw,
                        flop_bound_ms=t_fl, bound="hbm" if t_bw >= t_fl else "fma", roof_fraction=max(t_bw, t_fl) / ms)
        r["PC_over_P"] = r["PC"]["ms_per_call"] / r["P"]["ms_per_call"]
        r["C_over_P"] = r["C"]["ms_per_call"] / r["P"]["ms_per_call"]
        print(json.dumps({k: (v if not isinstance(v, dict) else v["ms_per_call"]) for k, v in r.items()}), flush=True)
        res["runs"].append(r)
        est.close()
        del est, P, Cc, d
        torch.cuda.empty_cache()
    res["card_after"] = card()
    return res


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001 -- the card line is informative, the run does not depend on it
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--ticks", type=int, default=40)
    ap.add_argument("--foot", action="store_true", help="foot-state handles (dekf_get_foot_window) instead of the 9-state getters")
    ap.add_argument("--foot-n", type=int, nargs="+", default=[16384, 65536])
    ap.add_argument("--box", action="store_true", help="state-constrained handles (dekf_get_constrained_window)")
    ap.add_argument("--cross", action="store_true", help="dekf_get_window_cross_cov against each kind's covariance getter")
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    import torch
    from decentralized_ekf_mhe_b200 import build, estimator, synth
    build.build()
    if not torch.cuda.is_available():
        raise SystemExit("window_probe needs a CUDA device")
    peaks = estimator.measure_peaks(0)
    if a.foot or a.box or a.cross:
        res = (cross_main if a.cross else box_main if a.box else foot_main)(a, torch, estimator, synth, peaks)
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
        print("card:", res["card"])
        return
    N, n, warm = 20, a.n, 64
    res = dict(card=card(), torch_device=torch.cuda.get_device_name(0), n=n, N=N, warmup_ticks=warm, calls=a.calls, peaks=peaks,
               flops_per_stage=FLOPS, cov_flops_per_stage=FLOPS_COV, runs=[])
    for vo_name, jitter in (("ragged", True), ("lockstep", False)):
        d = synth.make_stream(n, warm + 2 * a.ticks + 1, vo_jitter=jitter, device="cuda")
        vo = [bool(d["vo_flag"][s].any()) for s in range(d["gyro"].shape[0])]
        for precision in ("fp64", "fp32"):
            for mode, mname in ((0, "full"), (1, "incremental")):
                prm = estimator.robot_params("go1", ekf_rate=200, N=N, window_solve=mode)
                est = estimator.BatchedEstimator(prm, n, precision=precision)
                est.run(0, warm, {k: v[:warm] for k, v in d.items()}, vo[:warm])
                T = warm - 1
                w = torch.empty(N, 9, n, dtype=torch.float64, device="cuda")
                h = est._hd
                K = torch.zeros(1, dtype=torch.int32)
                call = lambda: h.check(h.L.dekf_get_window(h.h, C.c_void_p(w.data_ptr()), C.cast(K.data_ptr(), C.POINTER(C.c_int32))),
                                       "dekf_get_window")
                for _ in range(5):
                    call()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.calls):
                    call()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / a.calls
                n_vo = est.window_vo_count().double().mean().item()
                Kv = int(K.item())
                esize = 8 if precision == "fp64" else 4
                by = algorithmic_bytes(N, Kv, esize, mode == 0)
                fb, ff = algorithmic_flops(Kv, n_vo, mode == 0)
                t_bw = by * n / (peaks["copy_gbs"] * 1e9) * 1e3
                t_fl = (fb * n / (peaks["fp64_tflops"] * 1e12) + ff * n / (peaks[precision + "_tflops"] * 1e12)) * 1e3
                # tick with and without the getter, alternated
                tick = {"plain": [], "with_getter": []}
                for j in range(2 * a.ticks):
                    s = warm + j
                    store = estimator.robot_store.from_stream(d, s)
                    key = "with_getter" if j % 2 else "plain"
                    e0.record()
                    est.step(s, store)
                    if j % 2:
                        call()
                    e1.record()
                    torch.cuda.synchronize()
                    tick[key].append(e0.elapsed_time(e1))
                tick = {k: sorted(v)[len(v) // 2] for k, v in tick.items()}
                # covariance getter: [K][81][n] doubles
                P = torch.empty(N, 81, n, dtype=torch.float64, device="cuda")
                cov = lambda: h.check(h.L.dekf_get_window_cov(h.h, C.c_void_p(P.data_ptr()), C.cast(K.data_ptr(), C.POINTER(C.c_int32))),
                                      "dekf_get_window_cov")
                for _ in range(5):
                    cov()
                torch.cuda.synchronize()
                e0.record()
                for _ in range(a.calls):
                    cov()
                e1.record()
                torch.cuda.synchronize()
                cov_ms = e0.elapsed_time(e1) / a.calls
                n_vo_c = est.window_vo_count().double().mean().item()
                Kc = int(K.item())
                cby = cov_algorithmic_bytes(N, Kc, esize, mode == 0)
                cfb, cff = cov_algorithmic_flops(Kc, n_vo_c, mode == 0)
                c_bw = cby * n / (peaks["copy_gbs"] * 1e9) * 1e3
                c_fl = (cfb * n / (peaks["fp64_tflops"] * 1e12) + cff * n / (peaks[precision + "_tflops"] * 1e12)) * 1e3
                del P
                r = dict(vo=vo_name, precision=precision, window_solve=mname, T=T, K=Kv, mean_vo_rows=n_vo, ms_per_call=ms,
                         bytes_per_instance=by, double_flops_per_instance=fb, handle_flops_per_instance=ff,
                         hbm_bound_ms=t_bw, flop_bound_ms=t_fl, bound="hbm" if t_bw >= t_fl else "fma",
                         roof_fraction=max(t_bw, t_fl) / ms, tick_ms_median=tick,
                         device_bytes=est.device_bytes(), cov_K=Kc, cov_mean_vo_rows=n_vo_c, cov_ms_per_call=cov_ms,
                         cov_bytes_per_instance=cby, cov_double_flops_per_instance=cfb, cov_handle_flops_per_instance=cff,
                         cov_hbm_bound_ms=c_bw, cov_flop_bound_ms=c_fl, cov_bound="hbm" if c_bw >= c_fl else "fma",
                         cov_roof_fraction=max(c_bw, c_fl) / cov_ms)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
                est.close()
                del est
        del d
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("card:", res["card"])


if __name__ == "__main__":
    main()
