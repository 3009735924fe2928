#!/usr/bin/env python
"""Benchmark of the estimator hot path (BASELINE.json metric: EKF+MHE instance-steps/s at a 64K batch).

    python bench.py --gpus N --steps K --warmup W            # our arm (sm_100a kernels through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: CPU path on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed tick's results to DIR/*.npy

One "step" = one lock-step tick of every instance in the batch: EKF tick (+VO correct/replay when a VO
message is due) + MHE update(T) (kinematics, stage assembly, VO bound insertion, marginalisation, full
window solve, output).  Workload = BASELINE configs[1]: Go1, 65,536 instances per GPU, N=20, 200 Hz, fp64,
synthetic trot stream with 30 Hz VO at 40 ms latency (SURVEY.md 8d).  Instances shard over ranks with no
collective on the data path (weak scaling: 65,536 instances per GPU).

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ekf_mhe_instance_steps_per_s"
UNIT = "instance-steps/s"
WORKLOAD = "go1_ekf_mhe_65536x_N20_fp64"
FILL_STEPS = 24  # untimed ticks before the timed region at N = 20; fill_steps(N) = max(24, N + 4): the steady state T >= N


def fill_steps(N):
    """Untimed ticks that bring every instance to the steady state (window full, marginalisation active)."""
    return max(FILL_STEPS, N + 4)

# Exact operation tally of the committed algorithm (tests/hostsim/flopcount.cpp; mul and add counted
# separately, FMA = 2; tests/test_flop_tally.py keeps these in sync with the kernels)
FLOPS = dict(meas_update=486, propagate=407, propagate_vo=1049, meas_update_pp=597, propagate_pp=503, propagate_vo_pp=1103,
             ekf_predict=432, ekf_correct=641, ekf_vo_correct=450, assemble_go1=1401, solve_epilogue=30)


def algorithmic_work(N, n_vo_mean, elt=8, depth_mean=None, depth_vo_mean=None):
    """Per instance-step algorithmic (bytes, flops) of each kernel (DESIGN.md 5).  Tier A (full window re-solve every
    tick): `solve` sweeps N+1 stages.  Tier B (incremental): `solve` is ONE stage from the newest checkpoint, `resweep`
    (ticks that carry VO bounds) restarts `depth_mean` stages back, `depth_vo_mean` of which carry a VO row."""
    rec = 25 * elt
    io = 3 * 8 + 12 * 8 + 8  # gyro in, x + v_body out, status
    w = {}
    if depth_mean is None:
        # full re-sweep: P_pp is carried through the arrival stage only (the "_pp" figures), not through the other N - 1
        w["solve"] = (2 * 54 * elt + (N + 1) * rec + io,
                      (N + 1) * FLOPS["meas_update"] + N * FLOPS["propagate"] + n_vo_mean * (
                          FLOPS["propagate_vo"] - FLOPS["propagate"]) + (FLOPS["meas_update_pp"] - FLOPS["meas_update"]) + (
                          FLOPS["propagate_pp"] - FLOPS["propagate"]) + FLOPS["solve_epilogue"])
    else:
        # incremental sweep: every stage carries P_pp (any checkpoint may become the arrival cost)
        w["solve"] = ((54 + 54 + 16 + 18) * elt + io + 4,
                      FLOPS["meas_update_pp"] + FLOPS["propagate_pp"] + FLOPS["solve_epilogue"])
        w["resweep"] = ((54 + depth_mean * 54 + (depth_mean + 1) * 25) * elt + io + 4,
                        depth_mean * (FLOPS["meas_update_pp"] + FLOPS["propagate_pp"]) + depth_vo_mean * (
                            FLOPS["propagate_vo_pp"] - FLOPS["propagate_pp"]) + FLOPS["solve_epilogue"])
    w["ekf"] = (7 * 8 + 2 * 20 * elt + 26 * elt + 8 + 4 * 8 + 4, FLOPS["ekf_predict"] + FLOPS["ekf_correct"])
    w["assemble"] = (4 * elt + 7 * 8 + 24 * 8 + 4 * 8 + 1 + rec + 5 * 8 + 4 + 8, FLOPS["assemble_go1"])
    return w


KERNEL_NAMES = {"full": {"solve": "k_solve_tma", "ekf": "k_ekf", "assemble": "k_assemble"},
                "incremental": {"solve": "k_solve_incr", "resweep": "k_solve_incr_tma", "ekf": "k_ekf", "assemble": "k_assemble"}}


def ncu_traffic(kernel, n=65536):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` over `n` instances, from the committed
    ncu --set full capture of this workload (profiles/r02_traffic.json: bytes per instance of the captured launch), or None."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        ent = json.load(open(p)).get(kernel)
        return None if ent is None else ent["dram_bytes_per_instance"] * n
    except Exception:
        return None


def kernel_report(mode, work, pms, pcnt, n, hbm_peak, hbm_src, fma_peak, precision, extra_alg):
    """Per-kernel achieved GB/s and TFLOP/s from the event-pair times, and the roofline object of the dominant one."""
    kern = {}
    for name, (by, fl) in work.items():
        if pcnt.get(name, 0) == 0:
            continue
        dur = pms[name] / pcnt[name] * 1e-3
        kern[name] = {"kernel": KERNEL_NAMES[mode][name], "ms": dur * 1e3, "launches": pcnt[name], "total_ms": pms[name],
                      "gbs": by * n / dur / 1e9, "tflops": fl * n / dur / 1e12, "bytes_per_instance": by, "flops_per_instance": fl}
    tot = sum(v["total_ms"] for v in kern.values()) or 1.0
    dom = max(kern, key=lambda k: kern[k]["total_ms"]) if kern else "solve"
    kd = kern.get(dom, {"gbs": 0.0, "tflops": 0.0, "ms": 0.0, "total_ms": 0.0})
    t_hbm = work[dom][0] / (hbm_peak * 1e9)
    t_fma = work[dom][1] / (fma_peak * 1e12) if fma_peak > 0 else 0.0
    if t_fma >= t_hbm:
        roof = {"bound": "fp64" if precision == "fp64" else "fp32", "achieved": kd["tflops"], "peak": fma_peak,
                "unit": "TFLOP/s", "frac": kd["tflops"] / fma_peak if fma_peak else None}
    else:
        roof = {"bound": "hbm", "achieved": kd["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": kd["gbs"] / hbm_peak}
    alg = {"bytes_per_instance_step": work[dom][0], "flops_per_instance_step": work[dom][1]}
    alg.update(extra_alg)
    roof.update({
        "kernel": KERNEL_NAMES[mode][dom], "kernel_ms": kd["ms"], "kernel_share_of_step": kd["total_ms"] / tot,
        "kernel_ms_source": "CUDA event pair around every launch on the launching stream (dekf_profile_*), mean over a "
                            "separate tick-by-tick pass of the same workload, no host sync between launches",
        "traffic": ncu_traffic(KERNEL_NAMES[mode][dom], n),
        "hbm": {"achieved": kd["gbs"], "peak": hbm_peak, "frac": kd["gbs"] / hbm_peak, "peak_source": hbm_src},
        "fma": {"achieved": kd["tflops"], "peak": fma_peak, "frac": kd["tflops"] / fma_peak if fma_peak else None,
                "peak_source": "measured in this run (dekf_measure_fma_peak, non-tensor FMA)"},
        "algorithmic": alg, "all_kernels": kern})
    return roof


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                 getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                 getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        med = None
        if self.samples:
            s = sorted(self.samples)
            med = s[len(s) // 2]
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


DUMP_BYTES = 60 * 10**6  # array bytes --dump-outputs writes at most, summed over ranks (with the .npy headers: under 64 MB)


def dump_outputs(path, outs, lo, rank, world, seed=20240510):
    """Writes what the timed dekf_run call handed its caller for the last timed tick (quat, x, v_body, contact, status) as
    <path>/<name>.npy in float64, instances along the last axis, and the global index of every written instance as
    instance.npy.  Above DUMP_BYTES a fixed, seeded sample of the instances is written, the same in every run."""
    import numpy as np
    arrs = {k: v.numpy().astype(np.float64) for k, v in outs.items()}
    n = arrs["x"].shape[-1]
    per_instance = 8 * (1 + sum(a.size // n for a in arrs.values()))
    keep = min(n, DUMP_BYTES // world // per_instance)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(seed + rank).choice(n, keep, replace=False))
    arrs = {k: a[..., idx] for k, a in arrs.items()}
    arrs["instance"] = (lo + idx).astype(np.float64)
    os.makedirs(path, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for k, a in arrs.items():
        np.save(os.path.join(path, f"{k}{suffix}.npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def shared_config(n, world, N, precision, robot="go1", box=False, leg_odom_type=0, est_type=0, window_solve="full"):
    """The `config` object of the JSON line: a pure function of the workload, identical for our arm and the reference arm."""
    std = (robot == "go1" and n == 65536 and N == 20 and precision == "fp64" and not box and leg_odom_type == 0 and est_type == 0)
    return {"workload": WORKLOAD if std else f"{robot}_ekf_mhe_{n}x_N{N}_{precision}" + ("_box" if box else "") +
            ("_footstates" if leg_odom_type else "") + ("_kf" if est_type else ""),
            "robot": robot, "instances_per_gpu": n, "instances_total": n * world, "N": N, "rate_hz": 200,
            "vo": "30 Hz, 40 ms latency, lock-step arrival", "parallelism": f"instance-shard x{world}",
            "window_solve": window_solve, "est_type": est_type, "leg_odom_type": leg_odom_type, "v_box": bool(box),
            "cache": "per-step working set (window ring + inputs + per-tick outputs, > 300 MB at 65,536 instances) exceeds the 126 MB L2; "
                     "every step reads distinct input arrays and writes distinct output arrays"}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_run(N, K, W, min_seconds=5.0, max_seconds=150.0, mode="admm", ipt_min=64, seed=20240510):
    """The reference's CPU algorithm (oracle port) on the host cores: one instance at a time per thread, threads pinned,
    every thread stepping `ipt` instances through FILL + W warm-up + K timed steady-state ticks.  BASELINE.md section 2
    protocol: OSQP-style ADMM with a cold setup every tick, eps_abs = eps_rel = 1e-8, no wall-clock limit.  `ipt` is
    calibrated so that the timed region lasts at least `min_seconds` whatever K is (stable numbers), capped by
    `max_seconds` for the whole run.  Returns (instance-steps/s, timed seconds, instances, ipt, cores)."""
    from decentralized_ekf_mhe_b200 import synth
    from oracle import pyoracle as po
    cores = host_cores()
    po.pin_threads(True)
    fill = fill_steps(N)

    def params():
        if mode == "admm":
            return po.go1_params(N=N, solve_mode=2, time_limit=0.0, abs_tol=1e-8, relative_tol=1e-8)
        return po.go1_params(N=N, solve_mode=0)

    def run(ipt, ticks_timed, warm):
        n = cores * ipt
        S = fill + warm + ticks_timed
        st = synth.to_numpy(synth.make_stream(n, S, seed=seed))
        res, wall, busy = po.run_batch(st, params(), po.ekf_params(rate=200), nthreads=cores, t_steady=fill + warm, want=())
        return max(res["_busy_max"], 1e-9), n

    # calibration: 2 instances per thread x 6 timed ticks
    t_cal, n_cal = run(2, 6, 0)
    per_step = t_cal / (2 * 6)  # seconds per instance-step on the slowest thread
    # the calibration ticks are the slowest ones (cold caches, frequency ramp): 1.6x margin so that the timed region really
    # lasts min_seconds
    ipt = max(ipt_min, int(1.6 * min_seconds / max(K * per_step, 1e-9)) + 1)
    total_est = ipt * (fill + W + K) * per_step
    if total_est > max_seconds:
        ipt = max(1, int(max_seconds / ((fill + W + K) * per_step)))
    t, n = run(ipt, K, W)
    return n * K / t, t, n, ipt, cores


def batch1_latency(estimator, synth, device, precision, N, steps=300, window_solve=0):
    """Batch-1 lock-step tick latency: device time per tick (dekf_run over a resident stream, CUDA events) and host
    wall clock of one dekf_step_host call (pinned host buffers in and out, synchronised)."""
    import torch
    dev = torch.device("cuda", device)
    S = N + 8 + steps
    st = synth.make_stream(1, S, seed=777, device=dev, device_rng=True)
    vo = [bool(st["vo_flag"][s].any()) for s in range(S)]
    prm = estimator.robot_params("go1", ekf_rate=200, N=N, window_solve=window_solve)
    est = estimator.BatchedEstimator(prm, 1, device=device, precision=precision)
    cut = {k: v for k, v in st.items() if torch.is_tensor(v) and v.shape[0] == S}
    est.run(0, N + 8, cut, vo[:N + 8])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    est.run(N + 8, steps // 2, {k: v[N + 8:] for k, v in cut.items()}, vo[N + 8:N + 8 + steps // 2])
    e1.record()
    torch.cuda.synchronize()
    dev_us = e0.elapsed_time(e1) * 1e3 / (steps // 2)
    keys = ["gyro", "accel", "imu_time", "joint_pos", "joint_vel", "foot_force", "vo_quat", "vo_time_pre", "vo_time_now",
            "vo_rel_p", "vo_flag"]
    T = N + 8 + steps // 2
    host = {k: st[k][T:].cpu().pin_memory() for k in keys}
    out = {"quat": torch.empty(4, 1, dtype=torch.float64).pin_memory(), "x": torch.empty(9, 1, dtype=torch.float64).pin_memory(),
           "v_body": torch.empty(3, 1, dtype=torch.float64).pin_memory()}
    ts = []
    for j in range(S - T):
        d = {k: host[k][j] for k in keys}
        if not vo[T + j]:
            d["vo_flag"] = None
        t0 = time.perf_counter()
        est.step_host(T + j, d, out)
        ts.append(time.perf_counter() - t0)
    est.close()
    ts.sort()
    return {"device_us_per_tick": dev_us, "host_call_us_median": 1e6 * ts[len(ts) // 2], "host_call_us_p99": 1e6 * ts[int(len(ts) * 0.99)],
            "ticks": len(ts), "window_solve": "incremental" if window_solve else "full",
            "api": "dekf_step_host, n_instances=1 (k_fused: one launch per tick)"}


def _ref_sources_worker(job):
    """One process = one instance stepped through oracle/_ref/libref_nodes.so (the reference's own sources compiled against
    the stand-in Eigen/OSQP/rclcpp headers; its topic bus is process-global, hence processes, not threads)."""
    path, idx, t_steady = job
    import numpy as np
    from oracle import pyoracle as po, pyref as pr
    st = dict(np.load(path))
    prm = po.go1_params(N=int(st.pop("N")))
    rn = pr.RefNodes(prm, po.ekf_params(rate=200))
    S = st["gyro"].shape[0]
    t0 = 0.0
    for s in range(S):
        if s == t_steady:
            t0 = time.perf_counter()
        rn.tick_from_stream(st, s, idx)
    dt = time.perf_counter() - t0
    del rn
    return dt


def time_reference_sources(cores, N, ticks=40):
    """instance-steps/s of the reference's OWN sources (oracle/_ref/libref_nodes.so) with every host core, or None when the
    library did not travel.  Reported beside the port, never as the headline baseline: Eigen and OSQP are stand-ins there
    (dense eager linear algebra, exact KKT solve), so its speed says little about the real reference."""
    try:
        import tempfile
        from concurrent.futures import ProcessPoolExecutor
        import numpy as np
        from oracle import pyref as pr
        if not os.path.exists(pr._SO):
            return None
        from decentralized_ekf_mhe_b200 import synth
        t_steady = N + 4
        st = pr.quantize_stream(synth.to_numpy(synth.make_stream(cores, t_steady + ticks)))
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "stream.npz")
            np.savez(path, N=N, **st)
            import multiprocessing as mp
            with ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("spawn")) as ex:
                dts = list(ex.map(_ref_sources_worker, [(path, i, t_steady) for i in range(cores)]))
        return {"value": cores * ticks / max(dts), "unit": UNIT, "cores": cores, "kind": "reference sources + stand-in libraries",
                "sample": f"{cores} instances (one process each) x {ticks} steady-state ticks; exact KKT solve in the OSQP stand-in",
                "note": "correctness artefact (pins the oracle); NOT the headline baseline: the stand-in linear algebra is dense"}
    except Exception as e:  # never fail the bench on the optional leg
        return {"unavailable": repr(e)[:200]}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores.  The reference's own build
    (colcon + Eigen3 + OSQP + osqp-eigen + rclcpp) is impossible in this image; its sources do compile against stand-in
    headers into oracle/_ref/ (DESIGN.md 3), but with dense stand-in linear algebra and an exact KKT solve instead of OSQP
    that build is ~15x SLOWER than the real reference would be, so timing it would flatter our arm.  The headline of this
    arm is therefore the faster oracle port in its reference-faithful mode (BASELINE.md section 2: OSQP-style ADMM, cold
    setup every step, eps_abs = eps_rel = 1e-8, no wall-clock limit) with every host thread pinned, one instance at a time
    per thread; the compiled reference sources are timed beside it (`reference_sources`) for transparency.  A "step" is one
    tick of the bounded sample batch (cores x ipt instances); ipt >= 64 and the timed region lasts >= 5 s whatever --steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", args.gpus))
    K, W = args.steps, max(args.warmup, 3)
    N = args.N
    value, t, n, ipt, cores = cpu_reference_run(N, K, W, min_seconds=5.0, mode="admm", ipt_min=args.ref_instances_per_thread)
    sample = (f"{n} instances ({ipt}/thread, {cores} pinned threads) x {K} steady-state ticks after {fill_steps(N)} fill + {W} warm-up "
              f"ticks; oracle port, OSQP-style ADMM eps_abs=eps_rel=1e-8, cold setup every tick, time_limit=0; timed {t:.1f} s")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": 1e3 * t / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64" if args.precision == "fp64" else "f32", "data": "synthetic",
        "config": shared_config(args.instances, world, N, args.precision, args.robot, args.box, args.leg_odom_type, args.est_type,
                                args.window_solve),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    rs = time_reference_sources(min(cores, 16), N)
    if rs is not None:
        line["reference_sources"] = rs
    print(json.dumps(line))
    return 0


BOX = dict(v_box_enable=1, v_box_lo=(-0.45, -0.03, -0.015), v_box_hi=(0.55, 0.03, 0.015))  # binds in ~50 % of the PogoX steps


def bind_rank_to_host(local_rank, local_world):
    """One process per GPU: give every rank its own slice of the host cores -- the cores of its GPU's NUMA node when sysfs
    says which that is -- and prefer that node for the pinned buffers it allocates afterwards (first touch happens on these
    cores; set_mempolicy(MPOL_PREFERRED) when the node is allowed).  Returns what was done, for the JSON line."""
    info = {"cores": None, "numa_node": None, "mempolicy": None}
    try:
        allowed = sorted(os.sched_getaffinity(0))
        node = None
        try:
            import torch
            pr = torch.cuda.get_device_properties(local_rank)
            bdf = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            v = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
            node = v if v >= 0 else None
        except Exception:
            node = None
        pool = allowed
        if node is not None:
            try:
                cl = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
                cpus = set()
                for part in cl.split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
                near = [c for c in allowed if c in cpus]
                if len(near) >= 2:
                    pool = near
            except Exception:
                pass
        k = max(1, len(pool) // max(1, local_world))
        mine = pool[(local_rank * k) % len(pool):][:k] or pool
        os.sched_setaffinity(0, mine)
        info["cores"] = [mine[0], mine[-1], len(mine)]
        info["numa_node"] = node
        if node is not None:
            try:
                import ctypes
                libc = ctypes.CDLL(None, use_errno=True)
                mask = ctypes.c_ulong(1 << node)
                MPOL_PREFERRED = 1
                rc = libc.syscall(238, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(8 * ctypes.sizeof(mask)))
                info["mempolicy"] = "preferred" if rc == 0 else f"errno {ctypes.get_errno()}"
            except Exception as e:
                info["mempolicy"] = repr(e)[:60]
    except Exception as e:
        info["error"] = repr(e)[:80]
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=65536, help="instances per GPU")
    ap.add_argument("--N", type=int, default=20)
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    ap.add_argument("--robot", default="go1", choices=["go1", "cassie", "pogox"])
    ap.add_argument("--box", action="store_true", help="state constraints lo <= v_s <= hi on every window state (BASELINE config 4)")
    ap.add_argument("--leg-odom-type", type=int, default=0, choices=[0, 1])
    ap.add_argument("--est-type", type=int, default=0, choices=[0, 1])
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--window-solve", default="full", choices=["full", "incremental"],
                    help="full: re-sweep the whole window every tick (tier A, the reference's semantics); "
                         "incremental: restart at the first changed stage (tier B, bit-identical results)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the compact objects of BASELINE configs 3/4/5 and the ragged-VO stream")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-instances-per-thread", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last timed tick to DIR/<name>.npy (float64; the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from decentralized_ekf_mhe_b200 import build as b
    b.build()
    from decentralized_ekf_mhe_b200 import estimator, synth
    from decentralized_ekf_mhe_b200.sharding import env_rank, max_over_ranks, shard_range

    rank, local_rank, world = env_rank()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    binding = bind_rank_to_host(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    if world > 1:
        # NCCL (the contract's backend) carries only the barrier and the max-over-ranks of the device time; DEKF_BENCH_BACKEND=gloo
        # exists to tell a slow rank from an effect of the communicator itself (profiles/r02b_multigpu.md)
        # NVLS (NVLink SHARP multicast, which NCCL sets up from 4 GPUs on) is switched off for this communicator: with it three of
        # four ranks ran the SAME kernels 10 % slower (0.1075 vs 0.0978 ms per tick; 0.098 with gloo; independent processes 0.0975),
        # and an 8-byte all-reduce gains nothing from in-switch reduction.  NCCL_NVLS_ENABLE in the environment overrides.
        os.environ.setdefault("NCCL_NVLS_ENABLE", "0")
        if os.environ.get("DEKF_BENCH_BACKEND", "nccl") == "gloo":
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    W, K = max(args.warmup, 3), args.steps
    Ke = max(1, min(args.e2e_steps, K))
    n = args.instances  # per GPU (weak scaling)
    n_total = n * world
    lo, hi = shard_range(n_total, rank, world)
    assert hi - lo == n
    N = args.N
    FILL = fill_steps(N)
    robot = args.robot
    plain = not (args.box or args.leg_odom_type or args.est_type)  # the 9-state MHE: both solve modes exist
    base_over = dict(est_type=args.est_type, leg_odom_type=args.leg_odom_type, **(BOX if args.box else {}))
    S = FILL + W + K + 2 * (Ke + 8) + 20 + 24
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gen_stream(rb, nn, SS, jitter=False, seed=20240510 + 7919 * rank, amp=False):
        st = synth.make_stream(nn, SS, robot=rb, seed=seed, device=dev, device_rng=True, vo_jitter=jitter, amp_jitter=amp)
        vo = [bool(st["vo_flag"][s].any()) for s in range(SS)]
        return st, vo

    def sub(st, a, b_, SS):
        return {k: v[a:b_] for k, v in st.items() if torch.is_tensor(v) and v.shape[0] == SS}

    def step_outputs(est, kk, nn):
        """Per-tick result arrays of the timed region: every tick writes quat, x, v_body, contact, status."""
        ds, nl = est._hd.ds, est._hd.nl
        return {"quat": torch.empty(kk, 4, nn, dtype=torch.float64, device=dev), "x": torch.empty(kk, ds, nn, dtype=torch.float64, device=dev),
                "v_body": torch.empty(kk, 3, nn, dtype=torch.float64, device=dev), "contact": torch.empty(kk, nl, nn, dtype=torch.uint8, device=dev),
                "status": torch.empty(kk, nn, dtype=torch.int32, device=dev)}

    def device_pass(rb, nn, NN, precision, over, st, vo, SS, t0, kk, profile_ticks=0, keep=False, last=False):
        """kk ticks in one dekf_run call, inputs resident in HBM, every tick's results written to per-tick arrays, CUDA events
        on the launching stream, max over ranks; optionally a tick-by-tick pass of a fresh handle with an event pair around
        every launch (per-kernel device time).  last=True: res["last"] holds the results of the last tick on the host."""
        prm = estimator.robot_params(rb, ekf_rate=200, N=NN, **over)
        est = estimator.BatchedEstimator(prm, nn, device=local_rank, precision=precision)
        est.run(0, t0, sub(st, 0, t0, SS), vo[:t0])
        outs = step_outputs(est, kk, nn)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        timed = sub(st, t0, t0 + kk, SS)
        barrier()
        l0 = est.launch_count()
        ev0.record()
        est.run(t0, kk, timed, vo[t0:t0 + kk], out=outs, out_per_step=True)
        ev1.record()
        barrier()
        ms_rank = ev0.elapsed_time(ev1)
        ms = max_over_ranks(ms_rank)
        per_rank = [ms_rank]
        if world > 1:
            per_rank = [None] * world
            dist.all_gather_object(per_rank, ms_rank)
        res = dict(ms=ms, ms_per_rank=per_rank, launches=est.launch_count() - l0, checksum=float(outs["x"][:, 3].double().sum().item()),
                   finite=bool(torch.isfinite(outs["x"]).all().item()), bytes=est.device_bytes())
        if over.get("v_box_enable"):
            it, na = est.qp_info()
            res["factorisations_mean"] = float(it.double().mean())
            res["active_bounds_mean"] = float(na.double().mean())
        if last:
            res["last"] = {k: v[-1].cpu() for k, v in outs.items()}
        del outs
        if profile_ticks:
            Kp = min(kk, profile_ticks)
            est2 = estimator.BatchedEstimator(prm, nn, device=local_rank, precision=precision)
            est2.run(0, t0, sub(st, 0, t0, SS), vo[:t0])
            est2.profile(True)
            dsum = torch.zeros((), dtype=torch.float64, device=dev)
            vsum = torch.zeros((), dtype=torch.float64, device=dev)
            wsum = torch.zeros((), dtype=torch.float64, device=dev)
            nvo_ticks = 0
            incr = over.get("window_solve", 0) == 1
            for s_ in range(t0, t0 + Kp):
                est2.step(s_, estimator.robot_store.from_stream(st, s_, with_vo=vo[s_]))
                if rb != "pogox" or not over.get("v_box_enable"):
                    wsum += est2.window_vo_count().double().mean()  # VO rows in the window of THIS tick (flop tally operand)
                if incr and vo[s_]:
                    d_, v_ = est2.resweep_info()
                    dsum += d_.double().mean()
                    vsum += v_.double().mean()
                    nvo_ticks += 1
            pms, pcnt = est2.profile_read()
            est2.close()
            res.update(pms=pms, pcnt=pcnt, n_vo_mean=float(wsum.item()) / Kp, depth=float(dsum.item()) / max(nvo_ticks, 1),
                       depth_vo=float(vsum.item()) / max(nvo_ticks, 1), vo_tick_share=nvo_ticks / Kp)
        if keep:
            return est, res
        est.close()
        return None, res

    # ---- synthetic stream, resident in HBM before any timed region (each rank: its own instance range)
    t_gen = time.time()
    stream, vo_steps = gen_stream(robot, n, S)
    torch.cuda.synchronize()
    t_gen = time.time() - t_gen
    T0 = FILL + W

    sampler = ClockSampler(local_rank)
    sampler.start()
    mode = args.window_solve if plain else "full"
    other_mode = "full" if mode == "incremental" else "incremental"

    def over_for(md):
        o = dict(base_over)
        if plain:
            o["window_solve"] = 1 if md == "incremental" else 0
        return o

    est, main = device_pass(robot, n, N, args.precision, over_for(mode), stream, vo_steps, S, T0, K, profile_ticks=60 if plain else 0, keep=True,
                            last=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, main.pop("last"), lo, rank, world)
    other = None
    if plain:
        _, other = device_pass(robot, n, N, args.precision, over_for(other_mode), stream, vo_steps, S, T0, K, profile_ticks=60)
    ms_value, launches = main["ms"], main["launches"]
    value = n_total * K / (ms_value * 1e-3)
    T = T0 + K

    # ---- e2e: the same metric through the host-buffer entry point with pinned HOST streams: every tick's inputs are copied
    # H2D and every tick's results (quat, x_MHE, v_body, contact, status) are copied D2H inside the timed region.
    # Headline contract: dekf_run_host_f32io -- sensor streams as float32 (what the robot SDK delivers), results as float32;
    # time stamps, VO messages and ALL arithmetic double.  The all-double contract (dekf_run_host) is timed beside it.
    keys = ["gyro", "accel", "imu_time", "joint_pos", "joint_vel", "foot_force", "vo_quat", "vo_time_pre",
            "vo_time_now", "vo_rel_p"]
    F32 = estimator.BatchedEstimator.F32_KEYS
    rows = {k: (stream[k][0].numel() // n) for k in keys}
    ds_rows, nl = est._hd.ds, est._hd.nl
    Kw = 8  # untimed warm-up ticks of the host path (first call allocates the device staging and the copy streams)

    def host_slice(a, b_, f32):
        h = {k: stream[k][a:b_].reshape(b_ - a, rows[k], n).cpu() for k in keys}
        if f32:
            for k in F32:
                h[k] = h[k].float()
        h = {k: v.pin_memory() for k, v in h.items()}
        h["vo_flag"] = stream["vo_flag"][a:b_].cpu().pin_memory()
        return h

    def host_out(k, dt):
        return {"quat": torch.empty(k, 4, n, dtype=dt).pin_memory(), "x": torch.empty(k, ds_rows, n, dtype=dt).pin_memory(),
                "v_body": torch.empty(k, 3, n, dtype=dt).pin_memory(), "contact": torch.empty(k, nl, n, dtype=torch.uint8).pin_memory(),
                "status": torch.empty(k, n, dtype=torch.int32).pin_memory()}

    def e2e_pass(f32_in, f32_out, T, kk):
        fn = est.run_host_f32 if f32_in else est.run_host
        odt = torch.float32 if f32_out else torch.float64
        # every host buffer (warm-up and timed) is filled and pinned FIRST: staging ~1 GB on the host takes seconds, and a GPU /
        # PCIe link that idled that long spends the first 3-4 ms of the next call waking up (measured: tools/e2e_f32_probe.py,
        # 274 vs 244 us per tick over 100 ticks) -- the untimed warm-up call must run right before the timed one
        hst_w, hout_w = host_slice(T, T + Kw, f32_in), host_out(Kw, odt)
        hst, hout = host_slice(T + Kw, T + Kw + kk, f32_in), host_out(kk, odt)
        fn(T, Kw, hst_w, vo_steps[T:T + Kw], out=hout_w, out_per_step=True)
        T += Kw
        in_b = sum(rows[k] * (4 if (f32_in and k in F32) else 8) for k in keys[:6])
        h2d = sum(in_b * n + ((sum(rows[k] for k in keys[6:]) * 8 + 1) * n if vo_steps[T + j] else 0) for j in range(kk))
        d2h = (7 + ds_rows) * (4 if f32_out else 8) * n + nl * n + 4 * n
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.perf_counter()
        ev0.record()
        fn(T, kk, hst, vo_steps[T:T + kk], out=hout, out_per_step=True)
        chk = float(hout["x"][:, 3, 0].double().sum())  # read the results on the host
        ev1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = max_over_ranks(max(ev0.elapsed_time(ev1), wall * 1e3))  # device events vs host wall clock: the slower
        T += kk
        return T, {"value": n_total * kk / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d // kk, "d2h_bytes_per_step": d2h,
                   "steps": kk, "warmup_steps": Kw, "ms_per_step": ms / kk, "h2d_gbs": (h2d / kk) / (ms / kk * 1e-3) / 1e9,
                   "d2h_gbs": d2h / (ms / kk * 1e-3) / 1e9, "host_checksum": chk}

    Ke = max(1, min(Ke, (S - T - 2 * Kw - 44) // 2))
    T, e2e = e2e_pass(True, True, T, Ke)
    e2e["api"] = ("dekf_run_host_f32io: gyro, accel, joint_pos, joint_vel, foot_force travel as float32 pinned host streams (the robot SDK's "
                  "type), quat / x / v_body come back as float32; time stamps, VO messages and all arithmetic are double; H2D | kernels | "
                  "D2H pipelined over chunks of ticks, every tick's inputs copied in and results copied out")
    T, e2e64 = e2e_pass(False, False, T, Ke)
    e2e64["api"] = "dekf_run_host: all-double host streams and results (19.1 MB in + 8.9 MB out per tick at 65,536 Go1 instances)"
    # single-tick host path (dekf_step_host: copy in, step, copy out, sync) for comparison
    Ks = min(20, S - T)
    hs1 = host_slice(T, T + Ks, False)
    one_out = {k: v[0] for k, v in host_out(1, torch.float64).items() if k in ("quat", "x", "v_body")}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for j in range(Ks):
        d = {k: hs1[k][j] for k in keys}
        d["vo_flag"] = hs1["vo_flag"][j] if vo_steps[T] else None
        est.step_host(T, d, one_out)
        T += 1
    e2e["single_tick_host_call_ms"] = (time.perf_counter() - t0) * 1e3 / max(Ks, 1)
    est.close()
    del stream
    torch.cuda.empty_cache()

    # ---- ragged VO arrival (per-instance camera phase: every tick carries messages for some instances), both solve modes
    ragged = None
    configs = None
    if plain and not args.no_configs:
        Kr = min(K, 60)
        Sr = FILL + W + Kr
        st_r, vo_r = gen_stream(robot, n, Sr, jitter=True)
        ragged = {"vo": "30 Hz, 40 ms latency, per-instance camera phase (ragged arrival: every tick carries VO messages)", "steps": Kr}
        for md in ("full", "incremental"):
            _, r = device_pass(robot, n, N, args.precision, dict(window_solve=1 if md == "incremental" else 0), st_r, vo_r, Sr, FILL + W, Kr)
            ragged[md] = {"value": n_total * Kr / (r["ms"] * 1e-3), "unit": UNIT, "ms_per_step": r["ms"] / Kr, "finite": r["finite"]}
        del st_r
        torch.cuda.empty_cache()
    clocks = sampler.stop()

    # ---- BASELINE configs 3 / 4 / 5 as compact objects (the headline stays config 2)
    peaks = estimator.measure_peaks(local_rank) if rank == 0 or True else None
    if plain and not args.no_configs and robot == "go1":
        configs = {}
        cases = [("config3_cassie_fp64", "cassie", 65536, 20, "fp64", dict(window_solve=0), 40, False),
                 ("config3_cassie_fp32", "cassie", 65536, 20, "fp32", dict(window_solve=0), 40, False),
                 ("config4_pogox_box_16384", "pogox", 16384, 20, "fp64", dict(BOX), 12, False),
                 ("config5_go1_N100_shard_125000", "go1", 125000, 100, "fp64", dict(window_solve=0), 12, True),
                 ("go1_fp32", "go1", 65536, 20, "fp32", dict(window_solve=0), 40, False),
                 ("go1_kf_alternative", "go1", 65536, 20, "fp64", dict(est_type=1), 40, False),
                 ("go1_foot_states_16384", "go1", 16384, 20, "fp64", dict(leg_odom_type=1), 12, False)]
        for name, rb, nn, NN, prec, over, kk, amp in cases:
            try:
                fl = fill_steps(NN)
                SS = fl + 3 + kk
                st_c, vo_c = gen_stream(rb, nn, SS, jitter=(rb == "pogox"), amp=amp)
                _, r = device_pass(rb, nn, NN, prec, over, st_c, vo_c, SS, fl + 3, kk, profile_ticks=8 if "window_solve" in over else 0)
                ent = {"robot": rb, "instances_per_gpu": nn, "N": NN, "precision": prec, "value": nn * world * kk / (r["ms"] * 1e-3), "unit": UNIT,
                       "ms_per_step": r["ms"] / kk, "steps": kk, "finite": r["finite"], "device_bytes": r["bytes"]}
                if "pms" in r and r["pcnt"].get("solve", 0):
                    elt = 8 if prec == "fp64" else 4
                    by, flp = algorithmic_work(NN, r["n_vo_mean"], elt)["solve"]
                    dur = r["pms"]["solve"] / r["pcnt"]["solve"] * 1e-3
                    pk = peaks["fp64_tflops"] if prec == "fp64" else peaks["fp32_tflops"]
                    ent["roofline"] = {"kernel": "k_solve_tma", "kernel_ms": dur * 1e3, "bound": prec, "achieved": flp * nn / dur / 1e12,
                                       "peak": pk, "unit": "TFLOP/s", "frac": flp * nn / dur / 1e12 / pk,
                                       "flops_per_instance_step": flp, "bytes_per_instance_step": by}
                for k_ in ("factorisations_mean", "active_bounds_mean"):
                    if k_ in r:
                        ent[k_] = r[k_]
                if "factorisations_mean" in r:
                    # k_box_team: ~60 kflop per block-tridiagonal factorisation of the window (DESIGN.md 8); latency-bound
                    flp = 60e3 * r["factorisations_mean"]
                    ent["roofline"] = {"kernel": "k_box_team", "bound": "latency (sequential stage recursion)", "achieved": flp * nn / (r["ms"] / kk * 1e-3) / 1e12,
                                       "peak": peaks["fp64_tflops"], "unit": "TFLOP/s", "frac": flp * nn / (r["ms"] / kk * 1e-3) / 1e12 / peaks["fp64_tflops"],
                                       "flops_per_instance_step": flp, "note": "flops are an estimate (60 kflop per factorisation)"}
                configs[name] = ent
                del st_c
                torch.cuda.empty_cache()
            except Exception as e:  # a side object must not take the headline down
                configs[name] = {"unavailable": repr(e)[:200]}

    # pinned-host copy bandwidth of this box (the roofline of the e2e path): one large H2D and D2H, both directions at once
    pcie = None
    try:
        nb = 256 << 20
        hb, hb2 = torch.empty(nb, dtype=torch.uint8).pin_memory(), torch.empty(nb, dtype=torch.uint8).pin_memory()
        db, db2 = torch.empty(nb, dtype=torch.uint8, device=dev), torch.empty(nb, dtype=torch.uint8, device=dev)
        s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        best = 0.0
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s1):
                db.copy_(hb, non_blocking=True)
            with torch.cuda.stream(s2):
                hb2.copy_(db2, non_blocking=True)
            torch.cuda.synchronize()
            best = max(best, nb / (time.perf_counter() - t0) / 1e9)
        pcie = best
        del hb, hb2, db, db2
    except Exception:
        pcie = None
    e2e["pinned_copy_gbs_each_way_measured"] = pcie
    e2e["host_binding"] = binding

    # ---- batch-1 step latency (BASELINE metric, second half): one instance, lock-step tick
    lat = lat_o = None
    if rank == 0 and plain:
        lat = batch1_latency(estimator, synth, local_rank, args.precision, N, window_solve=1 if mode == "incremental" else 0)
        lat_o = batch1_latency(estimator, synth, local_rank, args.precision, N, window_solve=0 if mode == "incremental" else 1)

    line = None
    if rank == 0:
        hbm_peak, hbm_src = measured_peaks()
        elt = 8 if args.precision == "fp64" else 4
        fma_peak = peaks["fp64_tflops"] if args.precision == "fp64" else peaks["fp32_tflops"]

        def report(md, res):
            if md == "incremental":
                work = algorithmic_work(N, res["n_vo_mean"], elt, depth_mean=res["depth"], depth_vo_mean=res["depth_vo"])
                extra = {"tier": "B (incremental: restart the sweep at the first changed stage; bit-identical to tier A)",
                         "resweep_depth_mean_on_vo_ticks": res["depth"], "vo_rows_in_resweep_mean": res["depth_vo"],
                         "vo_tick_share": res["vo_tick_share"]}
            else:
                work = algorithmic_work(N, res["n_vo_mean"], elt)
                extra = {"tier": "A (full-window re-solve every step)", "vo_stages_in_window_mean": res["n_vo_mean"]}
            return kernel_report(md, work, res["pms"], res["pcnt"], n, hbm_peak, hbm_src, fma_peak, args.precision, extra)

        cfg = shared_config(n, world, N, args.precision, robot, args.box, args.leg_odom_type, args.est_type, mode)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_value / K, "ms_per_step_per_rank": [m / K for m in main["ms_per_rank"]], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if args.precision == "fp64" else "f32", "data": "synthetic",
            "config": cfg,
            "timed_region": {"api": "dekf_run, inputs resident in HBM", "outputs": "every tick writes quat, x, v_body, contact, status to "
                             "per-tick device arrays (out_per_step)", "checksum_vx": main["checksum"], "finite": main["finite"],
                             "fill_steps": FILL, "stream_gen_s": round(t_gen, 2), "vo_stream": "lock-step arrival (headline); the ragged "
                             "stream is reported under `vo_ragged`"},
            "e2e": e2e,
            "e2e_f64_io": e2e64,
            "gpu_launches": launches,
            "clocks": {k: clocks[k] for k in ("sm_mhz", "sm_max_mhz", "reasons")},
        }
        if plain:
            roof = report(mode, main)
            roof["measured_copy_gbs"] = peaks["copy_gbs"]
            # the whole step against its roofline (BASELINE north_star: "the slower of bytes-per-step over HBM bandwidth and
            # flops-per-step over FP64/FP32 peak"): algorithmic bytes / flops of ALL kernels of a tick over the timed ms_per_step
            # of the pipelined region -- in dekf_run the launches of consecutive ticks overlap, so this, not the duration of one
            # launch timed alone (`kernel_ms` above: 1.73 waves at 65,536 instances), is what the timed region achieves
            ak = roof.get("all_kernels", {})
            sb = sum(v["bytes_per_instance"] * v["launches"] for v in ak.values()) / max(1, max(v["launches"] for v in ak.values())) if ak else 0.0
            sf = sum(v["flops_per_instance"] * v["launches"] for v in ak.values()) / max(1, max(v["launches"] for v in ak.values())) if ak else 0.0
            step_s = ms_value / K * 1e-3
            t_h, t_f = sb * n / (hbm_peak * 1e9), (sf * n / (fma_peak * 1e12) if fma_peak else 0.0)
            roof["step"] = {"bytes_per_instance_step": sb, "flops_per_instance_step": sf, "ms_per_step": ms_value / K,
                            "bound": "hbm" if t_h >= t_f else ("fp64" if args.precision == "fp64" else "fp32"),
                            "hbm_gbs": sb * n / step_s / 1e9, "hbm_frac": sb * n / step_s / 1e9 / hbm_peak,
                            "tflops": sf * n / step_s / 1e12, "fma_frac": (sf * n / step_s / 1e12 / fma_peak) if fma_peak else None,
                            "frac": max(t_h, t_f) / step_s}
            line["roofline"] = roof
            line["latency_batch1"] = lat
            line["ekf_only"] = {"value": n_total / (roof["all_kernels"]["ekf"]["ms"] * 1e-3) if "ekf" in roof.get("all_kernels", {}) else None,
                                "unit": "EKF ticks/s", "note": "orien_ekf::timerCallback alone (k_ekf, event pairs, incl. the VO rewind/"
                                "replay ticks): the reference runs this filter as its own 500 Hz process"}
            line["full_resweep" if other_mode == "full" else "incremental"] = {
                "window_solve": other_mode, "value": n_total * K / (other["ms"] * 1e-3), "unit": UNIT, "ms_per_step": other["ms"] / K,
                "gpu_launches": other["launches"], "latency_batch1": lat_o, "roofline": report(other_mode, other)}
        else:
            line["roofline"] = {"bound": "latency", "achieved": None, "peak": None, "unit": "TFLOP/s", "frac": None, "traffic": None,
                                "note": "variant path (see DESIGN.md 8 / 9): no per-kernel tally"}
        if ragged is not None:
            line["vo_ragged"] = ragged
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            # the same protocol as the reference arm (bench.py --impl reference), bounded to ~cpu-seconds of timed work
            # (same sample size and duration as `--impl reference --steps 20 --warmup 3`: 16 pinned threads run at a higher clock in a
            # 6 s region than in a 13 s one -- 7.6e3 vs 5.4e3 measured on one box -- so the two legs must not differ in length)
            v, t, nn, ipt, cores = cpu_reference_run(N, 20, 3, min_seconds=5.0, mode="admm", ipt_min=args.ref_instances_per_thread)
            vd, td, _, _, _ = cpu_reference_run(N, 20, 3, min_seconds=2.0, max_seconds=20.0, mode="direct", ipt_min=8)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{nn} instances ({ipt}/thread, {cores} pinned threads) x 20 steady-state ticks; oracle port in reference-faithful "
                          f"mode (OSQP-style ADMM, cold setup every tick, eps_abs=eps_rel=1e-8, no time limit); timed {t:.1f} s",
                "direct_solve_value": vd,
                "direct_solve_note": "same port with the exact banded solve instead of ADMM (algorithmic CPU baseline)"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
