#!/usr/bin/env python
"""Wide batch engine (65 to 1,024 landmarks, covariances in HBM) against one streamed handle per filter.

For each (n, B) of the table below, Sigma totals 4.5 to 10 GB, far above the 126 MB of L2.  Inputs are device-resident
(step_known_dev), so the timed window holds the step kernels only.  --traj trajectories are simulated on the host and
repeated across the batch; every filter still has its own covariance.

Per size the JSON line reports
  - corrections/s and ms per step (batch timers, after --warmup steps);
  - bytes moved: passes over Sigma (sweep_count) x 16 N ld bytes (the padded rows the sweep reads and writes), plus the
    five rows of Sigma each correction reads;
  - that traffic's rate as a fraction of a device-to-device copy of the batch's Sigma (cudaMemcpyAsync via
    torch's copy_), timed in the same run;
  - the baseline: 32 streamed handles (EKF_SLAM(n, engine=ENGINE_STREAM), default settings) stepped one after the
    other on the same trajectories, as corrections/s;
  - a bit-identity spot check of two filters against streamed handles with set_carry_pending(False).

  python scripts/bench_wide_batch.py [--steps K] [--warmup W] [--sizes 65:32768,128:8192] [--out FILE]

Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [(65, 32768), (128, 8192), (256, 2048), (512, 1024), (1024, 296)]
BASELINE_HANDLES = 32


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], check=True,
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the numbers are still reported; say that the card could not be read
        return {"name": None, "power_limit": None, "error": str(e)}


def world_for(pkg, n):
    nx = max(d for d in range(1, int(np.sqrt(n)) + 1) if n % d == 0)
    return pkg.tracegen.grid_world(n // nx, nx, pitch=0.35)


def copy_rate(torch, nbytes, reps=3):
    """Bytes/s (read + write) of a device-to-device copy of nbytes."""
    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3
    del src, dst
    torch.cuda.empty_cache()
    return 2.0 * nbytes * reps / s


def run_size(pkg, torch, n, B, steps, warmup, traj, seed):
    T = warmup + steps
    tr = pkg.tracegen.simulate_known(world_for(pkg, n), min(traj, B), T, seed=seed)
    reps = -(-B // tr["xy"].shape[1])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (1, reps) + (1,) * (a.ndim - 2))[:, :B])  # noqa: E731
    tw, xy, vis = tile(tr["twists"]), tile(tr["xy"]), tile(tr["vis"])
    d_tw, d_xy, d_vis = (torch.from_numpy(a).cuda() for a in (tw, xy, vis))
    torch.cuda.synchronize()
    N = 3 + 2 * n
    ld = (N + 15) // 16 * 16
    bt = pkg.EKFBatch(B, n)

    def step(t):
        bt.step_known_dev(d_tw[t].data_ptr(), d_xy[t].data_ptr(), d_vis[t].data_ptr())

    for t in range(warmup):
        step(t)
    bt.sync()
    u0, s0 = bt.update_count, bt.sweep_count
    bt.timer_start()
    for t in range(warmup, T):
        step(t)
    ms = bt.timer_stop()
    corr, sweeps = bt.update_count - u0, bt.sweep_count - s0
    sweep_bytes = sweeps * 16 * N * ld
    gain_bytes = corr * 5 * 8 * N
    res = {
        "n": n, "B": B, "N": N, "ld": ld, "sigma_total_gb": round(B * N * ld * 8 / 1e9, 2),
        "steps": steps, "ms_per_step": round(ms / steps, 4), "corrections": int(corr),
        "corrections_per_s": round(corr / (ms / 1e3), 1), "sweeps": int(sweeps),
        "bytes_moved": int(sweep_bytes + gain_bytes), "bytes_per_s": round((sweep_bytes + gain_bytes) / (ms / 1e3), 1),
    }
    # bit-identity spot check: two filters against streamed handles with carry_pending off
    states = bt.states()
    same = True
    for b in (0, B - 1):
        f = pkg.EKF_SLAM(n, engine=pkg.ENGINE_STREAM)
        f.set_carry_pending(False)
        for t in range(T):
            f.prediction(tuple(tw[t, b]))
            f.measurement(xy[t, b], vis[t, b])
        same = same and np.array_equal(states[b], f.state) and np.array_equal(bt.sigma(b), f.sigma)
        f.close()
    res["bit_identical_to_streamed"] = bool(same)
    sigma_bytes = B * N * ld * 8
    bt.close()
    del d_tw, d_xy, d_vis
    torch.cuda.empty_cache()
    cr = copy_rate(torch, sigma_bytes)
    res["copy_bytes_per_s"] = round(cr, 1)
    res["fraction_of_copy_rate"] = round(res["bytes_per_s"] / cr, 4)
    # baseline: BASELINE_HANDLES streamed handles, default settings, stepped one after the other (host arrays)
    hs = [pkg.EKF_SLAM(n, engine=pkg.ENGINE_STREAM) for _ in range(BASELINE_HANDLES)]
    for t in range(warmup):
        for b, h in enumerate(hs):
            h.prediction(tuple(tw[t, b]))
            h.measurement(xy[t, b], vis[t, b])
    for h in hs:
        h.sync()
    c0 = sum(h.update_count for h in hs)
    t0 = time.perf_counter()
    for t in range(warmup, T):
        for b, h in enumerate(hs):
            h.prediction(tuple(tw[t, b]))
            h.measurement(xy[t, b], vis[t, b])
    for h in hs:
        h.sync()
    el = time.perf_counter() - t0
    bc = sum(h.update_count for h in hs) - c0
    for h in hs:
        h.close()
    res["baseline_corrections_per_s"] = round(bc / el, 1)
    res["speedup_vs_baseline"] = round(res["corrections_per_s"] / res["baseline_corrections_per_s"], 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--traj", type=int, default=1024, help="distinct simulated trajectories, repeated across the batch")
    ap.add_argument("--sizes", default=None, help="n:B,n:B,... (default: the table in the docstring)")
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    sizes = [tuple(int(v) for v in s.split(":")) for s in a.sizes.split(",")] if a.sizes else SIZES
    import torch

    import ekf_slam_ml_b200 as pkg
    if pkg.device_count() == 0 or not torch.cuda.is_available():
        raise SystemExit("bench_wide_batch.py needs a CUDA device")
    out = {"bench": "wide_batch", "gpu": gpu_info(), "steps": a.steps, "warmup": a.warmup, "traj": a.traj,
           "baseline_handles": BASELINE_HANDLES, "sizes": []}
    for n, B in sizes:
        out["sizes"].append(run_size(pkg, torch, n, B, a.steps, a.warmup, a.traj, a.seed))
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
