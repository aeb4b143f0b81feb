#!/usr/bin/env python
"""Cost of the batch NIS variants (ekf_batch_set_nis: the step kernels also accumulate every filter's normalised
innovation squared) against the plain step kernels, for each Sigma layout:

  tile       n = 20,    B = 65,536, known and unknown association (m_max = 12, as bench.py's batch_unknown)
  staircase  n = 33,    B = 16,384, known and unknown
  wide       n = 256,   B = 2,048 and n = 1,024, B = 296, known

Inputs are device-resident; --traj trajectories are simulated on the host and repeated across the batch.  Per size, after
--warmup steps with NIS off and on, --repeats rounds each time --steps steps with NIS off, then --steps with NIS on
(alternated in one process, same batch, consecutive input steps; the batch timers are CUDA events on the batch's
stream), then --calls calls of nis_dev (per-filter output and batch total, no reset).  The JSON line gives the medians
and the spread; "nis_overhead" is median(on) / median(off) - 1.

  python scripts/bench_nis.py [--steps K] [--calls C] [--repeats R] [--sizes 20:65536:known,...] [--out FILE]

Prints ONE JSON line; --out also writes it to a file (profiles/nis.json holds a B200 run).
"""
import argparse
import json
import os
import sys

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_consistency import gpu_info, world_for  # noqa: E402

SIZES = [(20, 65536, "known"), (20, 65536, "unknown"), (33, 16384, "known"), (33, 16384, "unknown"),
         (256, 2048, "known"), (1024, 296, "known")]
M_MAX = 12


def run_size(pkg, torch, n, B, kind, steps, warmup, calls, repeats, traj, seed):
    T = 2 * warmup + 2 * steps * repeats
    tg = pkg.tracegen
    if kind == "known":
        tr = tg.simulate_known(world_for(pkg, n), min(traj, B), T, seed=seed)
        keys = ("twists", "xy", "vis")
    else:
        tr = tg.simulate_unknown(tg.dense_world(n), min(traj, B), T, seed=seed, m_max=M_MAX)
        keys = ("twists", "meas", "count")
    reps = -(-B // tr["twists"].shape[1])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (1, reps) + (1,) * (a.ndim - 2))[:, :B])  # noqa: E731
    d = [torch.from_numpy(tile(tr[k])).cuda() for k in keys]
    d_pf = torch.empty((B, 4), dtype=torch.float64, device="cuda")
    d_out = torch.empty(4, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    bt = pkg.EKFBatch(B, n)
    if kind == "known":
        step = lambda t: bt.step_known_dev(*(x[t].data_ptr() for x in d))  # noqa: E731
    else:
        step = lambda t: bt.step_unknown_dev(*(x[t].data_ptr() for x in d), M_MAX)  # noqa: E731
    t = 0
    for on in (False, True):  # warm-up of both kernels
        bt.set_nis(on)
        for _ in range(warmup):
            step(t)
            t += 1
    ms = {False: [], True: []}
    nis_ms = []
    for _ in range(repeats):
        for on in (False, True):
            bt.set_nis(on)
            bt.sync()
            bt.timer_start()
            for _ in range(steps):
                step(t)
                t += 1
            ms[on].append(bt.timer_stop() / steps)
        bt.nis_dev(d_out.data_ptr(), d_pf.data_ptr())  # warm-up of the read-out
        bt.sync()
        bt.timer_start()
        for _ in range(calls):
            bt.nis_dev(d_out.data_ptr(), d_pf.data_ptr())
        nis_ms.append(bt.timer_stop() / calls)
    stats = pkg.consistency.anis_from_stats(d_out.cpu().numpy())
    bt.close()
    del d, d_pf
    torch.cuda.empty_cache()
    off, on, rd = float(np.median(ms[False])), float(np.median(ms[True])), float(np.median(nis_ms))
    return {
        "n": n, "B": B, "association": kind, "layout": "tile" if n == 20 else ("staircase" if n <= 64 else "wide"),
        "step_ms_nis_off": round(off, 4), "step_ms_nis_off_min_max": [round(min(ms[False]), 4), round(max(ms[False]), 4)],
        "step_ms_nis_on": round(on, 4), "step_ms_nis_on_min_max": [round(min(ms[True]), 4), round(max(ms[True]), 4)],
        "nis_overhead": round(on / off - 1.0, 4),
        "nis_dev_ms": round(rd, 4), "nis_dev_ms_min_max": [round(min(nis_ms), 4), round(max(nis_ms), 4)],
        "anis": stats["anis"], "scored": stats["count"], "nonfinite": stats["nonfinite"],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed SLAM steps per repeat and setting")
    ap.add_argument("--calls", type=int, default=50, help="timed nis_dev calls per repeat")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--traj", type=int, default=1024, help="distinct simulated trajectories, repeated across the batch")
    ap.add_argument("--sizes", default=None, help="n:B:known|unknown,... (default: the table in the docstring)")
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    sizes = [(int(s.split(":")[0]), int(s.split(":")[1]), s.split(":")[2]) for s in a.sizes.split(",")] if a.sizes \
        else SIZES
    import torch

    import ekf_slam_ml_b200 as pkg
    if pkg.device_count() == 0 or not torch.cuda.is_available():
        raise SystemExit("bench_nis.py needs a CUDA device")
    out = {"bench": "nis", "gpu": gpu_info(), "steps": a.steps, "calls": a.calls, "repeats": a.repeats,
           "warmup": a.warmup, "traj": a.traj, "m_max_unknown": M_MAX, "sizes": []}
    for n, B, kind in sizes:
        out["sizes"].append(run_size(pkg, torch, n, B, kind, a.steps, a.warmup, a.calls, a.repeats, a.traj, a.seed))
    out["gpu_after"] = gpu_info()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
