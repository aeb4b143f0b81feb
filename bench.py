#!/usr/bin/env python
"""bench.py — EKF measurement-updates/s on synthetic nurtlesim-shaped trajectories (BASELINE.json metric).

Headline workload (config.workload = "cfg3"): a Monte-Carlo batch of 65,536 independent filters x 20 landmark
slots PER GPU (weak scaling: filters are sharded over ranks with no data-path collective; ranks only
all-reduce error statistics), one "step" = prediction + measurement() for every filter (nuslam/src/slam.cpp:433-434).
Also measured at N=1 and reported in the same JSON line: the single large map (cfg4, n = 8,192, Sigma = 2.1 GB)
whose streamed rank-2 sweep is the clean HBM-roofline kernel.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ for the modules imported from it
ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "ekf_measurement_updates_per_sec"
UNIT = "updates/s"
N_SLOTS = 20
FILTERS_PER_GPU = 65536


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)  # first query is slow: take it now
            if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons"):
                pynvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception as e:  # NVML missing: report that, do not invent numbers
            self.nv = None
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.0002)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        if self._t:
            self._stop.set()
            self._t.join()
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ----------------------------------------------------------------------------- CPU legs (oracle/ as the checker)
def cpu_reference_known(cores, steps_inner, seed=1234, repeats=1):
    """The reference's own rigid2d::EKF_SLAM (oracle/_ref, built from the reference sources), one filter per host
    core, on the same kind of traces.  Returns (updates/s, description, kind)."""
    import _oracle
    import ekf_slam_ml_b200 as pkg
    tg = pkg.tracegen
    tr = tg.simulate_known(tg.dense_world(N_SLOTS), cores, steps_inner, seed=seed)
    tw = np.ascontiguousarray(tr["twists"].transpose(1, 0, 2))   # [f][t][2]
    xy = np.ascontiguousarray(tr["xy"].transpose(1, 0, 2))
    vis = np.ascontiguousarray(tr["vis"].transpose(1, 0, 2))
    L = _oracle.ref_lib()
    best = None
    if L is not None:
        upd = ctypes.c_int64()
        for _ in range(repeats):
            sec = L.ref_bench_known(N_SLOTS, cores, steps_inner, tw.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                    xy.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                    vis.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), ctypes.byref(upd), None)
            v = upd.value / sec
            best = v if best is None else max(best, v)
        return best, f"{cores} filters x {steps_inner} steps (prediction+measurement), n=20, one std::thread per filter; " \
                     f"reference ekf_slam.cpp compiled -O3 against the Armadillo stand-in over OpenBLAS (1 BLAS thread)", "reference"
    # no reference build on this box: the plain-C port, one python thread per filter (ctypes releases the GIL)
    Lo = _oracle.oracle_lib()
    filters = [_oracle.OracleEKF(N_SLOTS) for _ in range(cores)]
    counts = [0] * cores

    def run(f):
        counts[f] = Lo.oracle_run_known(filters[f].h, steps_inner, tw[f].ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                        xy[f].ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                        vis[f].ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
    t0 = time.perf_counter()
    th = [threading.Thread(target=run, args=(f,)) for f in range(cores)]
    [t.start() for t in th]
    [t.join() for t in th]
    sec = time.perf_counter() - t0
    return sum(counts) / sec, f"{cores} filters x {steps_inner} steps, plain-C O(N^2) port (oracle/ekf_oracle.c)", "port"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    steps_inner = 400
    vals = []
    for _ in range(args.warmup):
        cpu_reference_known(cores, steps_inner)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, sample, kind = cpu_reference_known(cores, steps_inner)
        vals.append(v)
    wall = time.perf_counter() - t0
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg3: Monte-Carlo batch of independent filters x 20 landmarks, known association "
                               "(bounded sample: one filter per host core)", "n_landmarks": N_SLOTS},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)



# ----------------------------------------------------------------------------- parity at the benchmarked sizes
PARITY_TOL = 1e-9  # scaled metric of tests/_oracle.py (state: max|d|/max(1,|x|); covariance: |d_ab| / max(|S_ab|, sqrt(S_aa S_bb)))


def scaled_rows_err(a, b, diag_b, row_ids, chunk=256):
    """Scaled covariance error over selected rows: a, b [k, N] (b = the checker), diag_b [N], row_ids [k]."""
    d = np.sqrt(np.abs(diag_b))
    worst = 0.0
    for i0 in range(0, a.shape[0], chunk):
        i1 = min(i0 + chunk, a.shape[0])
        scale = np.maximum(np.abs(b[i0:i1]), d[np.asarray(row_ids[i0:i1])][:, None] * d[None, :])
        np.maximum(scale, 1e-300, out=scale)
        worst = max(worst, float(np.max(np.abs(a[i0:i1] - b[i0:i1]) / scale)))
    return worst


def parity_cfg3(bt, tr, n, picks=64, seed=5):
    """After the timed steps: `picks` random filters of the batch against the plain-C oracle driven through the
    whole trajectory the batch went through (known association)."""
    import _oracle
    B = tr["twists"].shape[1]
    T = tr["twists"].shape[0]
    rng = np.random.default_rng(seed)
    ids = sorted(set([0, B - 1] + [int(v) for v in rng.integers(0, B, picks)]))
    states = bt.states()
    worst_s = worst_c = 0.0
    for b in ids:
        o = _oracle.OracleEKF(n)
        for t in range(T):
            o.prediction(*tr["twists"][t, b])
            o.measurement(tr["xy"][t, b], tr["vis"][t, b])
        worst_s = max(worst_s, _oracle.state_err(states[b], o.state))
        worst_c = max(worst_c, _oracle.sigma_err(bt.sigma(b), o.sigma))
    ok = bool(worst_s < PARITY_TOL and worst_c < PARITY_TOL)
    return {"ok": ok, "filters_checked": len(ids), "steps": int(T), "state_err": worst_s, "sigma_err": worst_c,
            "tol": PARITY_TOL, "checker": "oracle/ekf_oracle.c (plain-C restatement pinned to the reference build)"}


def parity_large_map(pkg, device, n_lm, tr, min_corrections=10, max_pending=None):
    """cfg4 size: a fresh streamed filter and the O(N^2) oracle through the init-only call and as many steps as it
    takes to pile up >= min_corrections corrections (they stay pending on the GPU and go through ONE multi-factor
    sweep when Sigma is read); state and the FULL covariance compared.  Also times the oracle (CPU baseline)."""
    import _oracle
    f = pkg.EKF_SLAM(n_lm, device=device)
    if max_pending:
        f.set_max_pending(max_pending)
    o = _oracle.OracleEKF(n_lm)
    N = 3 + 2 * n_lm
    done, t, cpu_s, cpu_n = 0, 0, 0.0, 0
    while done < min_corrections and t < tr["twists"].shape[0]:
        f.prediction(tuple(tr["twists"][t, 0]))
        f.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        o.prediction(*tr["twists"][t, 0])
        t0 = time.perf_counter()
        o.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        if t > 0:  # step 0 is the init-only call
            k = int(tr["vis"][t, 0].sum())
            cpu_s += time.perf_counter() - t0
            cpu_n += k
            done += k
        t += 1
    s0 = f.sweep_count
    st_err = _oracle.state_err(f.state, o.state)
    sig = f.sigma            # settles the pending factors: one sweep with P = pending corrections
    sweeps = f.sweep_count - s0
    ref = o.sigma
    c_err = scaled_rows_err(sig, ref, np.diag(ref).copy(), np.arange(N), chunk=128)
    f.close()
    ok = bool(st_err < PARITY_TOL and c_err < PARITY_TOL)
    par = {"ok": ok, "n_landmarks": n_lm, "state_dim": N, "corrections": done, "sweeps_at_readback": int(sweeps),
           "state_err": st_err, "sigma_err": c_err, "tol": PARITY_TOL, "entries_compared": int(N) * int(N),
           "checker": "oracle/ekf_oracle.c, O(N^2) form"}
    cpu = {"value": cpu_n / cpu_s if cpu_s > 0 else None, "unit": UNIT, "cores": 1, "kind": "port",
           "sample": f"{cpu_n} corrections at N={N}, plain-C O(N^2) port (the dense reference needs 2N^3 = "
                     f"{2.0 * N ** 3 / 1e12:.1f} TFLOP per correction and is intractable)"}
    return par, cpu


def parity_sharded(pkg, dist, local, n_lm, tr, min_corrections=10, sample_rows=None, seed=11):
    """cfg5: the row-sharded filter over the real NCCL ranks against the single-GPU streamed engine (one replica per
    rank, same inputs).  sample_rows = None: every owned row (full covariance); else that many rows in total."""
    from ekf_slam_ml_b200.sharded import ShardedEKF
    world, rank = dist.get_world_size(), dist.get_rank()
    f = ShardedEKF.from_process_group(n_lm, dist, local)
    g = pkg.EKF_SLAM(n_lm, device=local, engine=pkg.ENGINE_STREAM)
    N = 3 + 2 * n_lm
    done, t = 0, 0
    while done < min_corrections and t < tr["twists"].shape[0]:
        for obj in (f, g):
            obj.prediction(tuple(tr["twists"][t, 0]))
            obj.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        if t > 0:
            done += int(tr["vis"][t, 0].sum())
        t += 1
    st_err = float(np.max(np.abs(f.state - g.state) / np.maximum(1.0, np.abs(g.state))))
    r0, r1 = f.rows(0)
    if sample_rows is None:
        rows = np.arange(r0, r1, dtype=np.int64)
    else:
        rng = np.random.default_rng(seed + rank)
        k = max(1, sample_rows // world)
        rows = np.unique(np.concatenate([[r0, r1 - 1], rng.integers(r0, r1, k)])).astype(np.int64)
    diag = g.sigma_diag
    worst = 0.0
    for i0 in range(0, rows.size, 128):
        part = rows[i0:i0 + 128]
        worst = max(worst, scaled_rows_err(f.sigma_row_list(part), g.sigma_rows(part), diag, part))
    f.close()
    g.close()
    import torch
    e = torch.tensor([st_err, worst], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([float(rows.size)], dtype=torch.float64, device="cuda")
    dist.all_reduce(e, op=dist.ReduceOp.MAX)
    dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    st_err, worst = float(e[0].item()), float(e[1].item())
    return {"ok": bool(st_err < PARITY_TOL and worst < PARITY_TOL), "n_landmarks": n_lm, "state_dim": N,
            "corrections": done, "rows_compared": int(cnt.item()), "state_err": st_err, "sigma_err": worst,
            "tol": PARITY_TOL, "nccl_ranks": world,
            "checker": "single-GPU streamed engine (itself checked against the oracle at n = 8,192 in large_map.parity)"}


# ----------------------------------------------------------------------------- our arm
DUMP_STATES = 65536  # filters whose state is written by --dump-outputs (22.5 MB of float64 at n = 20)
DUMP_SIGMAS = 1024   # filters whose covariance is written (15.1 MB; all 65,536 would be 969 MB)


def dump_batch_outputs(bt, out_dir, seed=0):
    """What a caller of the timed path receives after its last step: the filters' states (bt.states()) and
    covariances (bt.sigma(b)), for all filters or a fixed, seeded sample of them, as float64 .npy files.  The
    *_filters.npy files hold the filter indices of each sample."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)
    st_ids = np.arange(bt.B) if bt.B <= DUMP_STATES else np.sort(rng.choice(bt.B, DUMP_STATES, replace=False))
    sg_ids = np.sort(rng.choice(bt.B, min(DUMP_SIGMAS, bt.B), replace=False))
    np.save(os.path.join(out_dir, "state.npy"), bt.states()[st_ids])
    np.save(os.path.join(out_dir, "state_filters.npy"), st_ids.astype(np.float64))
    np.save(os.path.join(out_dir, "sigma.npy"), np.stack([bt.sigma(int(b)) for b in sg_ids]))
    np.save(os.path.join(out_dir, "sigma_filters.npy"), sg_ids.astype(np.float64))


def cpu_reference_dense_scaling(pkg):
    """SURVEY.md section 8(d): the reference's own dense filter (oracle/_ref, one core) at growing map sizes, to show the
    cubic law that makes it intractable at cfg4 (2 N^3 flop per correction).  Whole-step time per correction."""
    import _oracle
    L = _oracle.ref_lib()
    if L is None:
        return None
    tg = pkg.tracegen
    rows = []
    for (nx, ny, steps) in ((5, 4, 120), (10, 10, 24), (25, 20, 4)):
        n = nx * ny
        tr = tg.simulate_known(tg.grid_world(nx, ny, pitch=0.5, n_slots=n, max_visible=0.7), 1, steps, seed=5)
        tw = np.ascontiguousarray(tr["twists"].transpose(1, 0, 2))
        xy = np.ascontiguousarray(tr["xy"].transpose(1, 0, 2))
        vis = np.ascontiguousarray(tr["vis"].transpose(1, 0, 2))
        upd = ctypes.c_int64()
        sec = L.ref_bench_known(n, 1, steps, tw.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                xy.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                vis.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), ctypes.byref(upd), None)
        rows.append({"n_landmarks": n, "state_dim": 3 + 2 * n, "corrections": int(upd.value), "steps": steps,
                     "ms_per_correction": 1e3 * sec / max(1, upd.value)})
    a, b = rows[-2], rows[-1]
    expo = float(np.log(b["ms_per_correction"] / a["ms_per_correction"]) / np.log(b["state_dim"] / a["state_dim"]))
    return {"kind": "reference", "cores": 1, "sizes": rows, "exponent_between_last_two": expo,
            "extrapolated_s_per_correction_at_N16387": 1e-3 * b["ms_per_correction"] * (16387.0 / b["state_dim"]) ** 3,
            "note": "reference ekf_slam.cpp, dense (I - K H) Sigma and A Sigma A^T GEMMs over single-thread OpenBLAS; the step's "
                    "prediction is included in the per-correction time"}



def large_map_leg(pkg, device, n_lm, timed_updates, peak_gbs, want_cpu):
    """cfg4: one filter, n_lm landmarks; streamed gain + sweep per correction."""
    tg = pkg.tracegen
    nx = int(round(np.sqrt(2 * n_lm)))
    ny = n_lm // nx
    assert nx * ny == n_lm, "large map expects n = nx*ny with nx = sqrt(2n)"
    w = tg.grid_world(nx, ny, pitch=0.5, n_slots=n_lm, max_visible=0.7)
    steps = 64
    tr = tg.simulate_known(w, 1, steps, seed=99)
    N = 3 + 2 * n_lm

    def timed(max_pending):
        # first call: initialise every landmark (ekf_slam.cpp:113-128), then a few warm-up steps, then ONE timed region
        # over whole SLAM steps until `timed_updates` corrections are done.  Factors stay pending across steps, so the
        # region ends with the flush that timer_stop() triggers (inside the timed region).
        f = pkg.EKF_SLAM(n_lm, device=device)
        if max_pending:
            f.set_max_pending(max_pending)
        t = 0
        while t < 3:
            f.prediction(tuple(tr["twists"][t, 0]))
            f.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
            t += 1
        f.sync()
        l0, s0 = f.launch_count, f.sweep_count
        done = 0
        f.timer_start()
        while t < steps and done < timed_updates:
            f.prediction(tuple(tr["twists"][t, 0]))
            f.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
            done += int(tr["vis"][t, 0].sum())
            t += 1
        ms = f.timer_stop()
        res = (ms, done, f.launch_count - l0, f.sweep_count - s0)
        f.close()
        return res

    env_p = int(os.environ["EKF_BENCH_MAX_PENDING"]) if os.environ.get("EKF_BENCH_MAX_PENDING") else None  # tuning aid
    sweep_ms_total, done, launches, n_sweeps = timed(env_p)
    ms_upd = sweep_ms_total / max(done, 1)
    alg_bytes = 16.0 * N * N
    out = {
        "workload": f"cfg4: single map, n={n_lm} landmarks (N={N}, Sigma {8.0 * N * N / 1e9:.3f} GB), known association, "
                    f"prediction + gain + streamed rank-2 sweep per correction",
        "value": 1e3 / ms_upd, "unit": UNIT, "updates_timed": done, "ms_per_update": ms_upd,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "k_large_sweep_mma<P> (time per sweep = whole step incl. predict + gains)",
                     "achieved": alg_bytes * n_sweeps / (sweep_ms_total * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                     "frac": alg_bytes * n_sweeps / (sweep_ms_total * 1e-3) / 1e9 / peak_gbs,
                     # ncu capture profiles/r2_prof_sweep_mma_raw.csv (P = 14): 2.235 GB read + 2.091 GB written per launch
                     "traffic": 4.326e9 if n_lm == 8192 else None,
                     "algorithmic_bytes_per_launch": alg_bytes, "sweeps": n_sweeps,
                     "updates_per_sweep": done / max(n_sweeps, 1),
                     "per_update_achieved": alg_bytes / (ms_upd * 1e-3) / 1e9,
                     "per_update_frac": alg_bytes / (ms_upd * 1e-3) / 1e9 / peak_gbs,
                     "note": "one launch moves Sigma once (16 N^2 B) and applies up to 14 pending corrections; per_update_* "
                             "is SURVEY.md's 16 N^2-per-correction convention and exceeds 1 for that reason"},
    }
    # untimed: parity at this size through the multi-factor sweep, against the O(N^2) oracle (which is the CPU baseline)
    par, cpu = parity_large_map(pkg, device, n_lm, tr)
    out["parity"] = par
    # the same leg with 20 corrections per sweep (ekf_set_max_pending): fewer passes over Sigma per correction, more
    # corrections/s, but the sweep is then bound by the FP64 pipe and no longer a copy - reported beside the default
    ms20, done20, launches20, sweeps20 = timed(20)
    par20, _ = parity_large_map(pkg, device, n_lm, tr, min_corrections=22, max_pending=20)
    out["deep_pending"] = {
        "max_pending": 20, "value": 1e3 * done20 / ms20, "unit": UNIT, "updates_timed": done20, "ms_per_update": ms20 / max(done20, 1),
        "gpu_launches": int(launches20), "sweeps": int(sweeps20), "updates_per_sweep": done20 / max(sweeps20, 1),
        "roofline": {"bound": "fp64 pipe (DMMA): 2 x 20 FMAs per element next to the copy", "unit": "GB/s", "peak": peak_gbs,
                     "achieved": alg_bytes * sweeps20 / (ms20 * 1e-3) / 1e9,
                     "frac": alg_bytes * sweeps20 / (ms20 * 1e-3) / 1e9 / peak_gbs,
                     "kernel": "k_large_sweep_mma_t<P, 256, 16, 4> (narrow tiles: the W fragments of 20 factors fit the registers)"},
        "parity": par20}
    if want_cpu:
        out["cpu_baseline"] = cpu
        dense = cpu_reference_dense_scaling(pkg)
        if dense is not None:
            out["cpu_baseline"]["dense_reference_scaling"] = dense
    return out


def sharded_map_leg(pkg, dist, local, n_lm, timed_updates, peak_gbs):
    """cfg5: one filter, n_lm landmarks, Sigma row-block-sharded over all ranks (per correction the two owning ranks
    store their partial W into every rank's exchange buffer from inside the correction kernel - or an NCCL all-reduce
    with EKF_SHARDED_EXCHANGE=nccl; K is formed locally on every rank).  Timed on the device, max over ranks."""
    from ekf_slam_ml_b200.sharded import ShardedEKF
    tg = pkg.tracegen
    world = dist.get_world_size()
    nx = int(round(np.sqrt(n_lm)))
    assert nx * nx == n_lm, "sharded map expects a square grid"
    w = tg.grid_world(nx, nx, pitch=0.5, n_slots=n_lm, max_visible=0.7)
    steps = 40
    tr = tg.simulate_known(w, 1, steps, seed=77)
    # untimed: parity over the real NCCL ranks, full covariance at the cfg4 size and sampled rows at this size
    n_small = 8192
    w_small = tg.grid_world(128, 64, pitch=0.5, n_slots=n_small, max_visible=0.7)
    par_small = parity_sharded(pkg, dist, local, n_small, tg.simulate_known(w_small, 1, 8, seed=99))
    par_full = parity_sharded(pkg, dist, local, n_lm, tr, sample_rows=1000)
    dist.barrier()
    f = ShardedEKF.from_process_group(n_lm, dist, local)
    if os.environ.get("EKF_BENCH_MAX_PENDING"):  # tuning aid: corrections per sweep (default 14)
        f.set_max_pending(int(os.environ["EKF_BENCH_MAX_PENDING"]))
    N = 3 + 2 * n_lm
    t = 0
    while t < 2:  # init-only call + one warm-up step
        f.prediction(tuple(tr["twists"][t, 0]))
        f.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        t += 1
    f.sync()
    dist.barrier()
    l0, s0 = f.launch_count, f.sweep_count
    done = 0
    # host-side preparation outside the timed region: the per-correction chain is ~20 us of GPU time, so python
    # conversions per step would otherwise be what is measured
    tw_l = [tuple(float(v) for v in tr["twists"][k, 0]) for k in range(steps)]
    xy_l = [np.ascontiguousarray(tr["xy"][k, 0]) for k in range(steps)]
    vis_l = [np.ascontiguousarray(tr["vis"][k, 0]) for k in range(steps)]
    cnt_l = [int(v.sum()) for v in vis_l]
    f.timer_start()
    while t < steps and done < timed_updates:  # one timed region; factors stay pending across steps
        f.prediction(tw_l[t])
        f.measurement(xy_l[t], vis_l[t])
        done += cnt_l[t]
        t += 1
    total_ms = pkg.sharding.allreduce_max(f.timer_stop(), dist, "cuda")  # timer_stop settles the pending factors first
    n_sweeps = f.sweep_count - s0
    ms_upd = total_ms / max(done, 1)
    rows = f.rows(0)
    per_gpu_bytes = 16.0 * N * N / world
    out = {
        "workload": f"cfg5: single map, n={n_lm} landmarks (N={N}, Sigma {8.0 * N * N / 1e9:.1f} GB) row-block-sharded over "
                    f"{world} GPUs; per correction: exchange of the partial W (2N fp64; {getattr(f, 'exchange', 'nccl all-reduce')}), "
                    f"K = W^T S^-1 formed on every rank, sweep of own rows",
        "value": 1e3 / ms_upd, "unit": UNIT, "updates_timed": done, "ms_per_update": ms_upd,
        "gpu_launches_rank0": int(f.launch_count - l0), "rows_rank0": list(rows), "w_exchange": getattr(f, "exchange", "nccl all-reduce"),
        "roofline": {"bound": "hbm", "kernel": "k_large_sweep_mma<P> on each rank's rows (time per sweep = whole step incl. "
                                                "prediction, gains and the W exchanges)",
                     "achieved": per_gpu_bytes * n_sweeps / (total_ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s per GPU",
                     "frac": per_gpu_bytes * n_sweeps / (total_ms * 1e-3) / 1e9 / peak_gbs, "traffic": None,
                     "algorithmic_bytes_per_launch_per_gpu": per_gpu_bytes, "sweeps": n_sweeps,
                     "updates_per_sweep": done / max(n_sweeps, 1),
                     "per_update_achieved": per_gpu_bytes / (ms_upd * 1e-3) / 1e9,
                     "per_update_frac": per_gpu_bytes / (ms_upd * 1e-3) / 1e9 / peak_gbs},
        "parity": {"ok": bool(par_small["ok"] and par_full["ok"]), "nccl_ranks": world,
                   "n8192_full_sigma": par_small, f"n{n_lm}_sampled_rows": par_full},
    }
    f.close()
    return out


def laser_leg(pkg, device, n_scans=8192):
    """(d) of the north star: 360-beam scans -> clusters -> circle fits -> classification, batched over scans."""
    import torch
    tg = pkg.tracegen
    sim = tg.TubeWorldSim(tg.default_world(), n_scans // 2, seed=31)
    scans = []
    for _ in range(2):
        for _ in range(21):
            sim.step_tick()
        scans.append(sim.laser_scan(360))
    scans = np.ascontiguousarray(np.concatenate(scans, axis=0))
    cf = pkg.CircleFitting(device=device, max_scans=n_scans, max_circles=16)
    ref_centers, ref_counts = cf.run_batch(scans)  # every cluster fitted (circleRegression on all of them)
    cf.set_centres_only(True)                      # approxCirclePositions(): accepted centres only
    centers, counts = cf.run_batch(scans)          # warm-up through the host path
    same = bool(np.array_equal(counts, ref_counts) and np.array_equal(np.nan_to_num(centers), np.nan_to_num(ref_centers)))
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        centers, counts = cf.run_batch(scans)
    e2e = reps * n_scans / (time.perf_counter() - t0)
    L = pkg._lib.load()
    d_scans = torch.from_numpy(scans).cuda()
    pkg.circle_fitting._check(L.circles_run_dev_f32(cf._ctx, d_scans.data_ptr(), n_scans))
    pkg.circle_fitting._check(L.circles_sync(cf._ctx))
    pkg.circle_fitting._check(L.circles_timer_start(cf._ctx))
    for _ in range(reps):
        pkg.circle_fitting._check(L.circles_run_dev_f32(cf._ctx, d_scans.data_ptr(), n_scans))
    ms = ctypes.c_float()
    pkg.circle_fitting._check(L.circles_timer_stop(cf._ctx, ctypes.byref(ms)))
    return {"workload": f"{n_scans} scans x 360 beams (float32), default 10-tube world: clustering + circle fit + classification",
            "scans_per_s_device": reps * n_scans / (ms.value * 1e-3), "scans_per_s_e2e": e2e,
            "circles_per_scan": float(counts.mean()), "kernel": "k_circles_scan<float>", "gpu_launches": reps,
            "mode": "approxCirclePositions (accepted centres only; clusters failing the inscribed-angle test skip the fit)",
            "centres_identical_to_full_fit": same}



def single_filter_leg(pkg, device, steps=400):
    """cfg1 / cfg2: ONE reference-sized filter (n = 20) at the node's cadence: prediction + measurement() (or
    data_association()) + pose read-back per step, through the C ABI (ctypes) and through the C++ facade, next to the
    reference's own class on one host core.  This is a LATENCY measurement (one launch sequence per call and a
    synchronising getter); the GPU is not expected to beat an 11 us CPU update here."""
    import subprocess
    import _oracle
    tg = pkg.tracegen
    tr = tg.simulate_known(tg.default_world(N_SLOTS), 1, steps + 21, seed=5)
    tu = tg.simulate_unknown(tg.default_world(N_SLOTS), 1, steps + 21, seed=5)
    out = {"workload": "cfg1 / cfg2: single filter, n = 20, default 10-tube world, one SLAM step per call sequence"}

    def run(obj, known, is_ref):
        kn = np.zeros(N_SLOTS, np.uint8)
        lat, upd = [], 0
        for t in range(steps + 21):
            t0 = time.perf_counter()
            if is_ref:
                obj.prediction(*(tr if known else tu)["twists"][t, 0])
            else:
                obj.prediction(tuple((tr if known else tu)["twists"][t, 0]))
            if known:
                obj.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
                k = int(tr["vis"][t, 0].sum())
            else:
                k = int(tu["count"][t, 0])
                if k:
                    obj.data_association(tu["meas"][t, 0, :k], kn)
            _ = obj.state[:3] if is_ref else obj._pose()
            if t > 20:
                lat.append(time.perf_counter() - t0)
                upd += k
        lat = np.array(lat)
        return {"us_per_step_mean": float(lat.mean() * 1e6), "us_per_step_median": float(np.median(lat) * 1e6),
                "updates_per_s": upd / float(lat.sum()), "updates_per_step": upd / len(lat)}

    for known in (True, False):
        f = pkg.EKF_SLAM(N_SLOTS, device=device)
        key = "known" if known else "unknown"
        out[key + "_c_abi"] = run(f, known, False)
        f.close()
        try:
            out[key + "_reference_cpu_1core"] = run(_oracle.RefEKF(N_SLOTS), known, True)
        except Exception as e:  # no reference build on this box
            out[key + "_reference_cpu_1core"] = {"unavailable": repr(e)}
    with tempfile.TemporaryDirectory() as tmp:  # built outside the tree, which may be read-only
        exe = os.path.join(tmp, "facade_latency")
        cmd = ["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "facade_latency.cpp"),
               "-o", exe, "-L" + os.path.join(ROOT, "ekf-slam-ml_b200"), "-lekfslam_b200", "-Wl,-rpath," + os.path.join(ROOT, "ekf-slam-ml_b200")]
        try:
            subprocess.run(cmd, check=True, capture_output=True, timeout=300)
            r = subprocess.run([exe, str(steps)], check=True, capture_output=True, text=True, timeout=300)
            out["cpp_facade"] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            out["cpp_facade"] = {"unavailable": repr(e)[:300]}
    return out


def large_map_unknown_leg(pkg, device, n_lm, peak_gbs, steps=24):
    """cfg4 'plus unknown association': the streamed engine's data_association() at n = 8,192 - per measurement one
    k_large_assoc launch over the known landmarks, then (if gated in) gain + ONE single-factor sweep, because the next
    measurement's distances need the corrected Sigma (ekf_slam.cpp:291-391)."""
    tg = pkg.tracegen
    nx = int(round(np.sqrt(2 * n_lm)))
    w = tg.grid_world(nx, n_lm // nx, pitch=0.5, n_slots=n_lm, max_visible=0.7)
    tr = tg.simulate_known(w, 1, steps + 4, seed=99)
    import _oracle
    f = pkg.EKF_SLAM(n_lm, device=device)
    N = 3 + 2 * n_lm
    # the map is built by the first measurement() call (all landmarks initialised, as in cfg4), then every step
    # associates the visible readings WITHOUT their labels against all n_lm known landmarks.  The first two such
    # steps run in lockstep with the oracle (untimed): association indices must be identical, state within tolerance.
    o = _oracle.OracleEKF(n_lm)
    f.prediction(tuple(tr["twists"][0, 0]))
    f.measurement(tr["xy"][0, 0], tr["vis"][0, 0])
    o.prediction(*tr["twists"][0, 0])
    o.measurement(tr["xy"][0, 0], tr["vis"][0, 0])
    known = np.ones(n_lm, np.uint8)
    known_o = np.ones(n_lm, np.uint8)
    meas_n = upd_n = 0
    ms_total = 0.0
    par_meas, par_same, par_margin = 0, True, np.inf
    for t in range(1, steps + 4):
        ids = np.flatnonzero(tr["vis"][t, 0])
        xy = tr["xy"][t, 0].reshape(-1, 2)[ids]
        f.prediction(tuple(tr["twists"][t, 0]))
        if t >= 4:
            f.sync()
            u0 = f.update_count
            f.timer_start()
        r = f.data_association(xy, known) if len(ids) else None
        if t >= 4:
            ms_total += f.timer_stop()
            meas_n += len(ids)
            upd_n += f.update_count - u0
        elif t <= 2:
            o.prediction(*tr["twists"][t, 0])
            if r is None:
                continue
            a, dmin, sec, _ = o.data_association(xy, known_o)
            par_meas += len(ids)
            par_same = par_same and bool(np.array_equal(r["assoc"], a))
            has = dmin < 10.0
            par_margin = min(par_margin, float(np.min(np.where(
                has, np.minimum.reduce([np.abs(dmin - 10.0), np.abs(dmin - 1.0), np.abs(sec - dmin)]), np.abs(sec - 10.0)))))
    st_err = None
    if par_meas:
        # the oracle stopped after step 2; compare against a second GPU filter stopped at the same point
        g = pkg.EKF_SLAM(n_lm, device=device)
        kg = np.ones(n_lm, np.uint8)
        for t in range(0, 3):
            g.prediction(tuple(tr["twists"][t, 0]))
            if t == 0:
                g.measurement(tr["xy"][0, 0], tr["vis"][0, 0])
            else:
                ids = np.flatnonzero(tr["vis"][t, 0])
                if len(ids):
                    g.data_association(tr["xy"][t, 0].reshape(-1, 2)[ids], kg)
        st_err = _oracle.state_err(g.state, o.state)
        g.close()
    f.close()
    alg = 16.0 * N * N
    return {"workload": f"cfg4 with unknown association: n={n_lm}, {meas_n / max(steps, 1):.1f} unlabelled measurements per step "
                        f"against {n_lm} known landmarks",
            "value": upd_n / (ms_total * 1e-3), "unit": UNIT, "measurements_per_s": meas_n / (ms_total * 1e-3),
            "ms_per_measurement": ms_total / max(meas_n, 1), "updates_timed": int(upd_n), "measurements_timed": int(meas_n),
            "parity": {"ok": bool(par_same and (st_err is None or st_err < PARITY_TOL)), "measurements_checked": par_meas,
                       "association_indices_identical": par_same, "smallest_decision_margin": par_margin,
                       "state_err": st_err, "tol": PARITY_TOL, "checker": "oracle/ekf_oracle.c in lockstep for the first two steps"},
            "roofline": {"bound": "hbm", "kernel": "k_large_sweep_p<1> (one sweep per associated measurement)", "unit": "GB/s",
                         "achieved": alg * upd_n / (ms_total * 1e-3) / 1e9, "peak": peak_gbs,
                         "frac": alg * upd_n / (ms_total * 1e-3) / 1e9 / peak_gbs, "traffic": None,
                         "note": "whole data_association() call incl. association kernels, gains and the host round trip "
                                 "for the outputs; 16 N^2 B per applied correction"}}


def scan_to_map_leg(pkg, device, B=8192, steps=12):
    """cfg2 batched: 360-beam scans -> clustering + circle fit + classification -> data_association, one robot per
    filter, everything on the device between the scan upload and the pose read-back."""
    import torch
    tg = pkg.tracegen
    s = tg.simulate_scans(tg.default_world(N_SLOTS), B, steps + 3, seed=21)
    cf = pkg.CircleFitting(device=device, max_scans=B, max_circles=16)
    cf.set_centres_only(True)
    bt = pkg.EKFBatch(B, N_SLOTS, device=device)
    M = 16
    total_scans = 0
    t_all = 0.0
    upd0 = 0
    for t in range(steps + 3):
        if t == 3:
            bt.sync()
            upd0 = bt.update_count
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        centers, counts = cf.run_batch(s["ranges"][t])      # host scans in, centres [B, 16, 2] + counts out
        meas = np.ascontiguousarray(centers[:, :M, :])
        cnt = np.minimum(counts, M).astype(np.int32)
        bt.step_unknown(np.ascontiguousarray(s["twists"][t]), meas, cnt, M)
        if t >= 3:
            total_scans += B
    bt.sync()
    t_all = time.perf_counter() - t0
    upd = bt.update_count - upd0
    out = {"workload": f"cfg2 batched: {B} robots, scan -> circles -> data_association per step (host scans in, host poses out)",
           "scans_per_s_e2e": total_scans / t_all, "updates_per_s": upd / t_all, "circles_per_scan": float(counts.mean()),
           "steps": steps, "ms_per_step": 1e3 * t_all / steps}
    bt.close()
    cf.close()
    return out


def batch_unknown_leg(pkg, device, B, steps, warmup):
    """cfg3, unknown-association variant: prediction + data_association (Mahalanobis gating) per filter and step."""
    import torch
    tg = pkg.tracegen
    M = 12
    T = steps + warmup
    tr = tg.simulate_unknown(tg.dense_world(N_SLOTS), B, T, seed=4242, m_max=M)
    bt = pkg.EKFBatch(B, N_SLOTS, device=device)
    d_tw = torch.from_numpy(np.ascontiguousarray(tr["twists"])).cuda()
    d_me = torch.from_numpy(np.ascontiguousarray(tr["meas"])).cuda()
    d_ct = torch.from_numpy(np.ascontiguousarray(tr["count"])).cuda()
    torch.cuda.synchronize()
    for t in range(warmup):
        bt.step_unknown_dev(d_tw[t].data_ptr(), d_me[t].data_ptr(), d_ct[t].data_ptr(), M)
    bt.sync()
    u0 = bt.update_count
    bt.timer_start()
    for t in range(warmup, T):
        bt.step_unknown_dev(d_tw[t].data_ptr(), d_me[t].data_ptr(), d_ct[t].data_ptr(), M)
    ms = bt.timer_stop()
    upd = bt.update_count - u0
    meas = int(tr["count"][warmup:].sum())
    out = {"workload": f"cfg3 unknown association: {B} filters x 20 slots, up to {M} unlabelled measurements per step",
           "value": upd / (ms * 1e-3), "unit": UNIT, "measurements_per_s": meas / (ms * 1e-3), "ms_per_step": ms / steps,
           "updates_per_step": upd / steps, "gpu_launches": steps}
    bt.close()
    return out


def device_sim_leg(pkg, device, B, steps, warmup):
    """SURVEY §8(f)-1: simulator -> filter without leaving the GPU (tube_world restatement feeding the fused step)."""
    tg = pkg.tracegen
    sim = pkg.TubeWorld(tg.dense_world(N_SLOTS), B, seed=777, device=device)
    bt = pkg.EKFBatch(B, N_SLOTS, device=device)
    sim.use_stream(bt.stream)
    p = sim.device_pointers()
    for _ in range(warmup + 1):
        sim.step_known()
        bt.step_known_dev(p["twists"], p["xy"], p["vis"])
    bt.sync()
    u0 = bt.update_count
    bt.timer_start()
    for _ in range(steps):
        sim.step_known()
        bt.step_known_dev(p["twists"], p["xy"], p["vis"])
    ms = bt.timer_stop()
    upd = bt.update_count - u0
    d = sim.download()
    err = bt.pose_error(d["truth"])
    oerr = np.sqrt(np.mean((d["odom"][:, :2] - d["truth"][:, :2]) ** 2, axis=0))
    # prediction() alone on the same twists (no landmark ever visible): what the motion model integrates from the
    # 10 Hz x10 twist -- replayed untimed on an identical generator (same seed => same trace)
    import torch
    sim2 = pkg.TubeWorld(tg.dense_world(N_SLOTS), B, seed=777, device=device)
    bp = pkg.EKFBatch(B, N_SLOTS, device=device)
    sim2.use_stream(bp.stream)
    p2 = sim2.device_pointers()
    blind = torch.zeros(B * N_SLOTS, dtype=torch.uint8, device=f"cuda:{device}")
    torch.cuda.synchronize()
    for _ in range(warmup + 1 + steps):
        sim2.step_known()
        bp.step_known_dev(p2["twists"], p2["xy"], blind.data_ptr())
    perr = bp.pose_error(sim2.download()["truth"])
    sim2.close()
    bp.close()
    out = {"workload": f"{B} robots simulated on the device (11 ticks + fake sensor per step) feeding the fused EKF step",
           "value": upd / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "gpu_launches": 2 * steps,
           "pose_rmse_xy": [float(np.sqrt(err[0] / err[3])), float(np.sqrt(err[1] / err[3]))],
           "odometry_rmse_xy": [float(oerr[0]), float(oerr[1])],
           "prediction_only_rmse_xy": [float(np.sqrt(perr[0] / perr[3])), float(np.sqrt(perr[1] / perr[3]))],
           "note": "SLAM vs prediction-only vs wheel odometry vs truth over the batch (the README's comparison, at "
                   "scale). The 100 Hz wheel odometer integrates the truth's own wheel increments, so it is exact "
                   "unless a robot collides (none does on this path); the filter's motion model sees the 10 Hz twist"}
    sim.close()
    bt.close()
    return out


def run_ours(args):
    import ekf_slam_ml_b200 as pkg
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    assert pkg.device_count() > local, "bench.py needs a CUDA device per rank (no CPU fallback)"
    peak_gbs, peak_src = measured_peaks()
    tg = pkg.tracegen
    B, n, K, W = args.filters, N_SLOTS, args.steps, args.warmup
    N = 3 + 2 * n
    T = W + K
    # ---- synthetic traces: filter index = rank*B + b, seeds differ per filter
    # 1 init-only step + T steps for the device-resident leg + 2 x T steps for the two end-to-end forms (one continuous run)
    tr = tg.simulate_known(tg.dense_world(n), B, 3 * T + 1, seed=2026, first_filter=rank * B, workers=host_cores())
    bt = pkg.EKFBatch(B, n, device=local)
    # step 0 of the trace is the node's init-only call; run it before anything is timed
    bt.step_known(np.ascontiguousarray(tr["twists"][0]), np.ascontiguousarray(tr["xy"][0]), np.ascontiguousarray(tr["vis"][0]))
    bt.sync()
    tw_h = pkg.PinnedBuffer((2 * T, B, 2), np.float64)
    xy_h = pkg.PinnedBuffer((2 * T, B, 2 * n), np.float64)
    vis_h = pkg.PinnedBuffer((2 * T, B, n), np.uint8)
    tw_h.array[...] = tr["twists"][T + 1:]
    xy_h.array[...] = tr["xy"][T + 1:]
    vis_h.array[...] = tr["vis"][T + 1:]
    poses_h = [pkg.PinnedBuffer((B, 3), np.float64) for _ in range(2)]
    upd_A = tr["vis"][1:T + 1].reshape(T, -1).sum(axis=1).astype(np.int64)
    upd_B = tr["vis"][T + 1:2 * T + 1].reshape(T, -1).sum(axis=1).astype(np.int64)
    upd_C = tr["vis"][2 * T + 1:].reshape(T, -1).sum(axis=1).astype(np.int64)

    def barrier():
        if dist:
            dist.barrier()

    import torch
    torch.cuda.set_device(local)
    # ---- leg A (`value`): inputs resident in HBM when the timed region starts
    d_tw = torch.from_numpy(np.ascontiguousarray(tr["twists"][1:T + 1])).cuda()
    d_xy = torch.from_numpy(np.ascontiguousarray(tr["xy"][1:T + 1])).cuda()
    d_vis = torch.from_numpy(np.ascontiguousarray(tr["vis"][1:T + 1])).cuda()
    torch.cuda.synchronize()

    def dev_step(t):
        bt.step_known_dev(d_tw[t].data_ptr(), d_xy[t].data_ptr(), d_vis[t].data_ptr())

    for t in range(W):
        dev_step(t)
    bt.sync()
    sampler = ClockSampler(local)
    barrier()
    torch.cuda.synchronize()
    l0 = bt.launch_count
    sampler.start()
    bt.timer_start()
    for t in range(W, T):
        dev_step(t)
    total_ms = bt.timer_stop()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop()
    launches = bt.launch_count - l0
    if args.dump_outputs and rank == 0:
        dump_batch_outputs(bt, args.dump_outputs)  # untimed; legs B and C below continue the same filters
    # The timed region holds exactly K launches of one kernel on one stream, so the average launch duration of
    # the dominant kernel is total_ms / K (CUDA events on the launching stream).
    updates_A = int(upd_A[W:T].sum())
    kern_ms_avg = total_ms / K
    upd_launch = float(upd_A[W:T].mean())
    t_ms = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    u_all = torch.tensor([updates_A], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(u_all, op=dist.ReduceOp.SUM)
    total_ms_max = float(t_ms.item())
    updates_all = float(u_all.item())
    value = updates_all / (total_ms_max * 1e-3)

    # ---- leg B (`e2e`): host (pinned) buffers through the public verbs; the H2D copy of each step's inputs and the
    # D2H read of its poses are inside the timed region.  The filters continue the same trajectories.
    # Two input forms, each with its own W warm-up + K timed steps: the dense arrays of measurement(), and the
    # fake_sensor message as published (visible markers only), which is what `e2e` quotes.
    def host_step_dense(t):
        bt.step_known(tw_h.array[t].ctypes.data, xy_h.array[t].ctypes.data, vis_h.array[t].ctypes.data)
        bt.poses_async(poses_h[t & 1])

    lists = [pkg.marker_list(xy_h.array[T + t], vis_h.array[T + t]) for t in range(T)]
    max_total = max(int(l[0][-1]) for l in lists)
    off_h = pkg.PinnedBuffer((T, B + 1), np.int32)
    ids_h = pkg.PinnedBuffer((T, max(max_total, 1)), np.uint8)
    pts_h = pkg.PinnedBuffer((T, max(max_total, 1), 2), np.float64)
    totals = []
    for t, (off, ids, pts) in enumerate(lists):
        off_h.array[t] = off
        ids_h.array[t, :len(ids)] = ids
        pts_h.array[t, :len(ids)] = pts
        totals.append(int(off[-1]))
    del lists

    def host_step_list(t):
        bt.step_known_sparse(tw_h.array[T + t].ctypes.data, off_h.array[t].ctypes.data, ids_h.array[t].ctypes.data,
                             pts_h.array[t].ctypes.data, totals[t])
        bt.poses_async(poses_h[t & 1])

    def timed(fn, upd, t0, t1):
        bt.sync()
        barrier()
        torch.cuda.synchronize()
        bt.timer_start()
        for t in range(t0, t1):
            fn(t)
        ms = bt.timer_stop()
        bt.sync()
        barrier()
        e_ms = torch.tensor([ms], dtype=torch.float64, device="cuda")
        u_b = torch.tensor([float(upd[t0:t1].sum())], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(u_b, op=dist.ReduceOp.SUM)
        return float(u_b.item()) / (float(e_ms.item()) * 1e-3), float(e_ms.item()) / (t1 - t0)

    for t in range(W):
        host_step_dense(t)
    dense_value, dense_ms = timed(host_step_dense, upd_B, W, T)
    for t in range(W):
        host_step_list(t)
    e2e_value, e2e_ms_step = timed(host_step_list, upd_C, W, T)
    h2d_dense = B * (2 * 8 + 2 * n * 8 + n)
    h2d = B * 2 * 8 + (B + 1) * 4 + float(np.mean(totals[W:T])) * 17
    d2h = B * 3 * 8

    # ---- untimed: parity of this rank's batch at the benchmarked size (64 random filters, whole trajectory)
    par3 = parity_cfg3(bt, tr, n)
    if dist:
        flag = torch.tensor([0.0 if par3["ok"] else 1.0, par3["state_err"], par3["sigma_err"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        par3.update(ok=bool(flag[0].item() == 0.0), state_err=float(flag[1].item()), sigma_err=float(flag[2].item()),
                    ranks=world)

    # ---- error statistics: the only inter-rank exchange of this workload (NCCL all-reduce of 4 doubles)
    err = bt.pose_error(np.ascontiguousarray(tr["truth"][3 * T][:, [0, 1, 2]]))
    e_t = torch.tensor(err, dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(e_t, op=dist.ReduceOp.SUM)
    err = e_t.cpu().numpy()

    # ---- roofline of the dominant kernel (ekf_fused_tile_kernel<false>: the only kernel inside the timed region)
    step_bytes = B * (2.0 * 8 * N * N)                      # dense Sigma in + out, once per filter and step
    conv_bytes = 16.0 * N * N * upd_launch                  # SURVEY.md §8(d): 16 N^2 per measurement-update
    tiled = (n == 20)
    # bytes one filter-step really moves: the 9,088-B block (Sigma as 15 DMMA fragments + robot rows + state) in and out,
    # plus its inputs (twist 16 B, 2n readings, n flags) and the init flag in / out
    stored_bytes = B * (2.0 * 9088 + 16 + 17 * n + 8) if tiled else None
    roof = {
        "bound": "hbm", "kernel": "ekf::tile::ekf_fused_tile_kernel<false>" if tiled else "ekf_fused_sym_kernel<0>",
        "unit": "GB/s", "peak": peak_gbs, "peak_source": peak_src,
        "achieved": step_bytes / (kern_ms_avg * 1e-3) / 1e9,
        "frac": step_bytes / (kern_ms_avg * 1e-3) / 1e9 / peak_gbs,
        # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel at this batch size, from the committed
        # ncu --set full capture (profiles/r2_prof_fused_tile_raw.csv: 619.4 MB read + 536.9 MB written); not re-measured here
        "traffic": 1.156e9 if (B == FILTERS_PER_GPU and tiled) else None,
        "algorithmic_bytes_per_launch": step_bytes,
        "stored_bytes_per_launch": stored_bytes,
        "physical_achieved": stored_bytes / (kern_ms_avg * 1e-3) / 1e9 if stored_bytes else None,
        "physical_frac": stored_bytes / (kern_ms_avg * 1e-3) / 1e9 / peak_gbs if stored_bytes else None,
        "note": "unit = one filter-step (prediction + all of the step's corrections with Sigma resident in registers). "
                "algorithmic bytes = 16 N^2 B = one read + one write of the dense Sigma the reference keeps; the kernel "
                "stores Sigma symmetric (15 DMMA accumulator fragments of the landmark block + 3 robot rows, 1,092 of "
                "1,849 entries), so the bytes it really moves (stored_bytes, physical_*; ncu traffic agrees) are 40 % fewer. "
                "per_update_* uses SURVEY.md's 16 N^2 per correction and exceeds 1 because the step's corrections share "
                "one pass over Sigma. Next to HBM the kernel is held by the FP64 pipe (DMMA + DFMA, ~60 % busy inside the "
                "correction loop) with three resident warps per SM sub-partition (168 registers each)",
        "per_update_achieved": conv_bytes / (kern_ms_avg * 1e-3) / 1e9,
        "per_update_frac": conv_bytes / (kern_ms_avg * 1e-3) / 1e9 / peak_gbs,
        "updates_per_launch": upd_launch, "kernel_ms": kern_ms_avg,
    }
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg3: Monte-Carlo batch, 65,536 independent filters x 20 landmark slots per GPU, "
                               "known association (prediction + measurement per step), nurtlesim-shaped circle trajectories, "
                               "20-tube world", "filters_per_gpu": B, "n_landmarks": n, "state_dim": N,
                   "l2": "inputs larger than L2 (Sigma + state batch = %.0f MB per step)" % (B * 9088.0 / 1e6 if tiled else B * 8.0 * N * N / 1e6),
                   "updates_per_step_per_gpu": upd_launch},
        "clocks": clocks,
        # headline end-to-end figure: the argument form of the reference's measurement(mat, vector<bool>, ...) - dense
        # [B,2n] readings + [B,n] visible flags from pinned host buffers, poses read back every step.  The same step fed
        # with the fake_sensor message as published (visible markers only) is reported beside it.
        "e2e": {"value": dense_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_dense), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": dense_ms,
                "input": "dense [B,2n] readings + [B,n] visible flags + twists [B,2], pinned host buffers, "
                         "ekf_batch_step_known + ekf_batch_get_poses_async per step (PCIe-bound: 23.3 MB per step)",
                "marker_list": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "ms_per_step": e2e_ms_step,
                                "input": "marker list (visible markers only: twists [B,2], CSR offsets, ids, xy; built on the "
                                         "host outside the timed region), ekf_batch_step_known_sparse"}},
        "gpu_launches": int(launches),
        "roofline": roof,
        "pose_rmse": {"x": float(np.sqrt(err[0] / err[3])), "y": float(np.sqrt(err[1] / err[3])),
                      "theta": float(np.sqrt(err[2] / err[3])), "filters": int(err[3])},
    }
    if rank == 0 and world == 1:
        cores = host_cores()
        v, sample, kind = cpu_reference_known(cores, 1500)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
        if not args.skip_large:
            bt.close()
            del d_tw, d_xy, d_vis
            torch.cuda.empty_cache()
            line["large_map"] = large_map_leg(pkg, local, args.large_n, args.large_updates, peak_gbs, want_cpu=True)
            line["large_map_unknown"] = large_map_unknown_leg(pkg, local, args.large_n, peak_gbs)
            line["single_filter"] = single_filter_leg(pkg, local)
            line["scan_to_map"] = scan_to_map_leg(pkg, local)
            line["batch_unknown"] = batch_unknown_leg(pkg, local, B, K, W)
            line["laser"] = laser_leg(pkg, local)
            line["device_sim"] = device_sim_leg(pkg, local, B, K, W)
    if world > 1 and not args.skip_large:
        # cfg5 needs every rank: free the batch first (Sigma shard = 51.2 GB / world per GPU)
        bt.close()
        del d_tw, d_xy, d_vis
        torch.cuda.empty_cache()
        sm = sharded_map_leg(pkg, dist, local, args.sharded_n, args.sharded_updates, peak_gbs)
        line["sharded_map"] = sm
    # parity summary: every leg that ran carries its own check; a mismatch makes the run fail (rc != 0)
    parity = {"cfg3": par3}
    if "large_map" in line:
        parity["cfg4"] = line["large_map"]["parity"]
        if "deep_pending" in line["large_map"]:
            parity["cfg4_20_per_sweep"] = line["large_map"]["deep_pending"]["parity"]
    if "sharded_map" in line:
        parity["cfg5"] = line["sharded_map"]["parity"]
        parity["nccl_ranks"] = world
    parity["ok"] = bool(all(v["ok"] for k, v in parity.items() if isinstance(v, dict)))
    line["parity"] = parity
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    if not parity["ok"]:
        sys.stderr.write("bench.py: PARITY MISMATCH at a benchmarked size: %s\n" % json.dumps(parity))
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--filters", type=int, default=FILTERS_PER_GPU, help="filters per GPU (cfg3 = 65536)")
    ap.add_argument("--large-n", type=int, default=8192)
    ap.add_argument("--large-updates", type=int, default=240)
    ap.add_argument("--skip-large", action="store_true")
    ap.add_argument("--only-large", action="store_true", help="profiling aid: run just the cfg4 leg")
    ap.add_argument("--only-laser", action="store_true", help="profiling aid: run just the laser front-end leg")
    ap.add_argument("--only-sharded", action="store_true", help="development aid (under torchrun): just the cfg5 leg")
    ap.add_argument("--only-small", action="store_true", help="development aid: single_filter, large_map_unknown, scan_to_map")
    ap.add_argument("--sharded-n", type=int, default=40000, help="cfg5 landmarks (square number), N>1 only")
    ap.add_argument("--sharded-updates", type=int, default=96)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the headline leg, write its filters' states and a seeded sample of "
                         "their covariances to DIR/*.npy (float64, under 64 MB; rank 0's batch)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.only_large or args.only_laser or args.only_sharded
                              or args.only_small):
        ap.error("--dump-outputs writes the headline leg's outputs: it cannot be combined with --impl reference "
                 "or --only-*")
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.only_large:
        import ekf_slam_ml_b200 as pkg
        print(json.dumps(large_map_leg(pkg, 0, args.large_n, args.large_updates, measured_peaks()[0], want_cpu=False)))
    elif args.only_laser:
        import ekf_slam_ml_b200 as pkg
        print(json.dumps(laser_leg(pkg, 0)))
    elif args.only_sharded:
        import torch
        import torch.distributed as dist
        import ekf_slam_ml_b200 as pkg
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        out = sharded_map_leg(pkg, dist, local, args.sharded_n, args.sharded_updates, measured_peaks()[0])
        if dist.get_rank() == 0:
            print(json.dumps(out), flush=True)
        dist.barrier()
        dist.destroy_process_group()
    elif args.only_small:
        import ekf_slam_ml_b200 as pkg
        print(json.dumps({"single_filter": single_filter_leg(pkg, 0),
                          "large_map_unknown": large_map_unknown_leg(pkg, 0, args.large_n, measured_peaks()[0]),
                          "scan_to_map": scan_to_map_leg(pkg, 0)}))
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
