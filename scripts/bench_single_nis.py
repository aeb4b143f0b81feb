#!/usr/bin/env python
"""Cost of the single filter's NIS variants (ekf_set_nis: measurement() / data_association() also score the normalised
innovation squared of their corrections) against the plain kernels, on one filter with NIS alternated off and on:

  fused     n = 20: one SLAM-node step through ctypes, host clock around work that ends in a synchronise:
            known association   prediction + measurement + pose read (slam.cpp:433-434),
            unknown association prediction + data_association + pose read (unknown_data_assoc.cpp:414-415);
  streamed  n = 8,192: ms per landmark correction, CUDA events on the filter's stream around --corr corrections per
            measurement() (carry_pending on, so the time includes the sweeps the corrections need);
  read-out  the host latency of one ekf_nis call (synchronises) on each filter.

Per case, after --warmup steps with NIS off and on, --repeats rounds each time --steps steps with NIS off, then --steps
with NIS on (same filter, consecutive input steps).  The JSON line gives the medians and the min / max over the
repeats; "nis_overhead" is median(on) / median(off) - 1.

  python scripts/bench_single_nis.py [--steps K] [--repeats R] [--large-n N] [--corr C] [--out FILE]

Prints ONE JSON line; --out also writes it to a file (profiles/single_nis.json holds a B200 run).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_consistency import gpu_info  # noqa: E402

M_MAX = 12


def _summary(ms, key):
    off, on = float(np.median(ms[False])), float(np.median(ms[True]))
    return {f"{key}_nis_off": round(off, 5), f"{key}_nis_off_min_max": [round(min(ms[False]), 5), round(max(ms[False]), 5)],
            f"{key}_nis_on": round(on, 5), f"{key}_nis_on_min_max": [round(min(ms[True]), 5), round(max(ms[True]), 5)],
            "nis_overhead": round(on / off - 1.0, 4)}


def _readout_us(f, calls):
    f.nis()
    t0 = time.perf_counter()
    for _ in range(calls):
        f.nis()
    return (time.perf_counter() - t0) / calls * 1e6


def run_fused(pkg, kind, steps, warmup, repeats, calls, seed):
    n, tg = 20, pkg.tracegen
    T = 2 * warmup + 2 * steps * repeats
    f = pkg.EKF_SLAM(n, engine=pkg.ENGINE_FUSED)
    if kind == "known":
        tr = tg.simulate_known(tg.dense_world(n), 1, T, seed=seed)
        tw, xy, vis = (np.ascontiguousarray(tr[k][:, 0]) for k in ("twists", "xy", "vis"))

        def step(t):
            f.prediction((tw[t, 0], tw[t, 1]))
            f.measurement(xy[t], vis[t])
            f.getStateX(), f.getStateY(), f.getStateTheta()
    else:
        tr = tg.simulate_unknown(tg.dense_world(n), 1, T, seed=seed, m_max=M_MAX)
        tw, meas, count = tr["twists"][:, 0], tr["meas"][:, 0], tr["count"][:, 0]
        known = np.zeros(n, np.uint8)
        meas_t = [np.ascontiguousarray(meas[t, :int(count[t])]) for t in range(T)]

        def step(t):
            f.prediction((tw[t, 0], tw[t, 1]))
            f.data_association(meas_t[t], known)
            f.getStateX(), f.getStateY(), f.getStateTheta()
    t = 0
    for on in (False, True):
        f.set_nis(on)
        for _ in range(warmup):
            step(t)
            t += 1
    ms = {False: [], True: []}
    for _ in range(repeats):
        for on in (False, True):
            f.set_nis(on)
            f.sync()
            t0 = time.perf_counter()
            for _ in range(steps):
                step(t)
                t += 1
            ms[on].append((time.perf_counter() - t0) / steps * 1e3)
    res = {"engine": "fused", "n": n, "association": kind, **_summary(ms, "step_ms"),
           "ekf_nis_us": round(_readout_us(f, calls), 2)}
    r = f.nis()
    res.update({"anis": r["anis"], "scored": r["count"], "nonfinite": r["nonfinite"]})
    return res


def run_streamed(pkg, n, corr, steps, warmup, repeats, calls, seed):
    rng = np.random.default_rng(seed)
    f = pkg.EKF_SLAM(n, engine=pkg.ENGINE_STREAM)
    xy0 = rng.uniform(-3.0, 3.0, 2 * n)
    f.prediction((0.0, 0.0))
    f.measurement(xy0, np.ones(n, np.uint8))  # initialises the map
    f.sync()

    def step():
        vis = np.zeros(n, np.uint8)
        vis[rng.choice(n, corr, replace=False)] = 1
        f.prediction((0.001, 0.002))
        f.measurement(xy0 + rng.normal(0.0, 0.01, 2 * n), vis)

    for on in (False, True):
        f.set_nis(on)
        for _ in range(warmup):
            step()
    ms = {False: [], True: []}
    for _ in range(repeats):
        for on in (False, True):
            f.set_nis(on)
            f.sync()
            f.timer_start()
            for _ in range(steps):
                step()
            ms[on].append(f.timer_stop() / (steps * corr))
    res = {"engine": "stream", "n": n, "association": "known", "corrections_per_call": corr,
           **_summary(ms, "ms_per_correction"), "ekf_nis_us": round(_readout_us(f, calls), 2)}
    r = f.nis()
    res.update({"anis": r["anis"], "scored": r["count"], "nonfinite": r["nonfinite"]})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed fused steps per repeat and setting")
    ap.add_argument("--large-steps", type=int, default=10, help="timed streamed measurement() calls per repeat and setting")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--calls", type=int, default=200, help="timed ekf_nis calls")
    ap.add_argument("--large-n", type=int, default=8192)
    ap.add_argument("--corr", type=int, default=28, help="corrections per streamed measurement() (two sweeps of 14)")
    ap.add_argument("--seed", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import ekf_slam_ml_b200 as pkg
    if pkg.device_count() == 0:
        raise SystemExit("bench_single_nis.py needs a CUDA device")
    out = {"bench": "single_nis", "gpu": gpu_info(), "steps": a.steps, "large_steps": a.large_steps,
           "repeats": a.repeats, "warmup": a.warmup, "calls": a.calls, "m_max_unknown": M_MAX, "cases": []}
    for kind in ("known", "unknown"):
        out["cases"].append(run_fused(pkg, kind, a.steps, a.warmup, a.repeats, a.calls, a.seed))
    out["cases"].append(run_streamed(pkg, a.large_n, a.corr, a.large_steps, min(a.warmup, 3), a.repeats, a.calls,
                                     a.seed))
    out["gpu_after"] = gpu_info()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
