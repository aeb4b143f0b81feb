#!/usr/bin/env python
"""Cost of the batch consistency read-out (ekf_batch_nees_dev: pose and landmark NEES of every filter, read from the
covariance in place) beside the batch's SLAM step, for each Sigma layout:

  tile       n = 20,    B = 65,536
  staircase  n = 33,    B = 16,384
  wide       n = 256,   B = 2,048 and n = 1,024, B = 296 (the sizes of scripts/bench_wide_batch.py)

Inputs are device-resident; --traj trajectories are simulated on the host and repeated across the batch.  Per size, after
--warmup steps, the batch timers (CUDA events on the batch's streams) time --steps SLAM steps, then --calls calls of
nees_dev with per-filter output and landmark truth, both repeated --repeats times; the JSON line gives the median and the
spread of each.  "bytes_read" is what the read-out needs from HBM: per filter the six pose entries, three entries of
each landmark block, the state, the init flag, the known list and the truth (pose and per-filter landmarks), plus the
per-filter output it writes; the achieved rate is that over the median call time.  The batches' covariances (0.6 to
4.5 GB) do not fit the 126 MB L2, but one read-out touches only a few percent of them, so part of what it reads may
still sit in L2 from the step before; the steps are not interleaved with the calls to keep each figure clean.

  python scripts/bench_consistency.py [--steps K] [--calls C] [--repeats R] [--sizes 20:65536,...] [--out FILE]

Prints ONE JSON line; --out also writes it to a file (profiles/consistency.json holds a B200 run).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [(20, 65536), (33, 16384), (256, 2048), (1024, 296)]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], check=True,
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:  # the numbers are still reported; say that the card could not be read
        return {"name": None, "error": str(e)}


def world_for(pkg, n):
    if n <= 33:
        return pkg.tracegen.dense_world(n)
    nx = max(d for d in range(1, int(np.sqrt(n)) + 1) if n % d == 0)
    return pkg.tracegen.grid_world(n // nx, nx, pitch=0.35)


def read_bytes(n, B):
    per_filter = 8 * (6 + 3 * n + 3 + 2 * n) + 4 + n + 8 * (3 + 2 * n) + 8 * 3
    return B * per_filter


def run_size(pkg, torch, n, B, steps, warmup, calls, repeats, traj, seed):
    T = warmup + steps * repeats
    w = world_for(pkg, n)
    tr = pkg.tracegen.simulate_known(w, min(traj, B), T, seed=seed)
    reps = -(-B // tr["xy"].shape[1])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (1, reps) + (1,) * (a.ndim - 2))[:, :B])  # noqa: E731
    tw, xy, vis, truth = tile(tr["twists"]), tile(tr["xy"]), tile(tr["vis"]), tile(tr["truth"])
    d_tw, d_xy, d_vis, d_truth = (torch.from_numpy(a).cuda() for a in (tw, xy, vis, truth))
    nt = min(w.n_tubes, n)
    lt = np.full((B, n, 2), np.nan)
    lt[:, :nt, 0], lt[:, :nt, 1] = w.tubes_x[:nt], w.tubes_y[:nt]
    d_lt = torch.from_numpy(lt).cuda()
    d_pf = torch.empty((B, 3), dtype=torch.float64, device="cuda")
    d_out = torch.empty(8, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    bt = pkg.EKFBatch(B, n)
    step = lambda t: bt.step_known_dev(d_tw[t].data_ptr(), d_xy[t].data_ptr(), d_vis[t].data_ptr())  # noqa: E731
    for t in range(warmup):
        step(t)
    t = warmup
    step_ms, nees_ms = [], []
    for _ in range(repeats):
        bt.sync()
        bt.timer_start()
        for _ in range(steps):
            step(t)
            t += 1
        step_ms.append(bt.timer_stop() / steps)
        last = d_truth[t - 1].data_ptr()
        bt.nees_dev(last, d_out.data_ptr(), d_lt.data_ptr(), 2 * n, d_pf.data_ptr())  # warm-up of this shape
        bt.sync()
        bt.timer_start()
        for _ in range(calls):
            bt.nees_dev(last, d_out.data_ptr(), d_lt.data_ptr(), 2 * n, d_pf.data_ptr())
        nees_ms.append(bt.timer_stop() / calls)
    stats = pkg.consistency.anees_from_stats(d_out.cpu().numpy())
    bt.close()
    del d_tw, d_xy, d_vis, d_truth, d_lt, d_pf
    torch.cuda.empty_cache()
    nb = read_bytes(n, B)
    med_step, med_nees = float(np.median(step_ms)), float(np.median(nees_ms))
    return {
        "n": n, "B": B, "layout": "tile" if n == 20 else ("staircase" if n <= 64 else "wide"),
        "step_ms": round(med_step, 4), "step_ms_min_max": [round(min(step_ms), 4), round(max(step_ms), 4)],
        "nees_ms": round(med_nees, 4), "nees_ms_min_max": [round(min(nees_ms), 4), round(max(nees_ms), 4)],
        "nees_over_step": round(med_nees / med_step, 4),
        "bytes_read": int(nb), "bytes_per_s": round(nb / (med_nees / 1e3), 1),
        "pose_anees": stats["pose_anees"], "landmark_anees": stats["landmark_anees"],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed SLAM steps per repeat")
    ap.add_argument("--calls", type=int, default=50, help="timed nees_dev calls per repeat")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--traj", type=int, default=1024, help="distinct simulated trajectories, repeated across the batch")
    ap.add_argument("--sizes", default=None, help="n:B,n:B,... (default: the table in the docstring)")
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    sizes = [tuple(int(v) for v in s.split(":")) for s in a.sizes.split(",")] if a.sizes else SIZES
    import torch

    import ekf_slam_ml_b200 as pkg
    if pkg.device_count() == 0 or not torch.cuda.is_available():
        raise SystemExit("bench_consistency.py needs a CUDA device")
    out = {"bench": "consistency", "gpu": gpu_info(), "steps": a.steps, "calls": a.calls, "repeats": a.repeats,
           "warmup": a.warmup, "traj": a.traj, "sizes": []}
    for n, B in sizes:
        out["sizes"].append(run_size(pkg, torch, n, B, a.steps, a.warmup, a.calls, a.repeats, a.traj, a.seed))
    out["gpu_after"] = gpu_info()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
