#!/usr/bin/env python
"""Tuning Q and R with one batch: every filter carries its own noise (EKFBatch.set_noise), so one EKFBatch of K groups x
M robots on TubeWorld sweeps a whole Q x R grid with one launch per step, and the device-side consistency read-outs
score every grid point.

The sweep runs report.py's world (dense_world(20), n = 20: the tile engine) for --steps SLAM steps.  The grid is
q = q_theta = q_x = q_y in QS times r = r_range = r_bearing in RS (16 points, from the reference's q = 1e-4, r = 0.01
towards more process and less measurement noise, which is where report.py's consistency table points).  Group g holds
robots g, g + K, g + 2K, ... (one simulator seed for the whole batch).  Per group it reports, from the per-filter
outputs of nis() and nees():
  ANIS (dof 2) and the pose ANEES (dof 3) and landmark ANEES (dof 2), each with its 95 % chi^2 interval, and the pose
  RMSE (x, y, theta) against the simulator's truth.

It also times the step with the default kernels against the NOISE variants set to the reference values, for the tile
(n = 20, B = 65,536), staircase (n = 33, B = 16,384) and wide (n = 256, B = 2,048) engines: --repeats rounds of --steps
steps with the default kernels, then --steps with the NOISE variant, alternated on one batch with device-resident
inputs (CUDA events on the batch's stream).

  python scripts/noise_sweep.py [--robots-per-point M] [--steps T] [--out profiles/noise_sweep.json]

Prints ONE JSON line; --out also writes it to a file.  Needs a CUDA device.
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

QS = [1e-4, 4e-4, 1.6e-3, 6.4e-3]
RS = [1e-2, 2.5e-3, 6.25e-4, 1.5625e-4]
TIMING = [(20, 65536), (33, 16384), (256, 2048)]


def grid():
    return np.array([[q, q, q, r, r] for q in QS for r in RS])


def sweep(pkg, M, steps, seed):
    cs = pkg.consistency
    g = grid()
    K = len(g)
    B = K * M
    world = pkg.tracegen.dense_world(20)
    n = world.n_slots
    sim = pkg.TubeWorld(world, B, seed=seed)
    bt = pkg.EKFBatch(B, n)
    rows = g[np.arange(B) % K]
    bt.set_noise(rows[:, :3], rows[:, 3:])
    bt.set_nis(True)
    sim.use_stream(bt.stream)
    p = sim.device_pointers()
    for _ in range(steps):
        sim.step_known()
        bt.step_known_dev(p["twists"], p["xy"], p["vis"])
    bt.sync()
    truth = sim.download()["truth"]
    nt = min(world.n_tubes, n)
    lm_truth = np.full((n, 2), np.nan)
    lm_truth[:nt] = np.stack([world.tubes_x[:nt], world.tubes_y[:nt]], axis=1)
    ni = bt.nis(per_filter=True)
    ne = bt.nees(truth, lm_truth, per_filter=True)
    est = bt.poses()[:, [1, 2, 0]]
    out = []
    for k in range(K):
        m = np.arange(B) % K == k
        st = np.array([ni["nis_sum"][m].sum(), ni["nis_sq_sum"][m].sum(), ni["nis_count"][m].sum(),
                       ni["nis_nonfinite"][m].sum()])
        a = cs.anis_from_stats(st)
        pose = ne["pose_nees"][m]
        runs = int(np.isfinite(pose).sum())
        lm_sum, lm_cnt = float(ne["landmark_nees_sum"][m].sum()), int(ne["landmark_nees_count"][m].sum())
        d = est[m] - truth[m]
        dth = np.arctan2(np.sin(d[:, 2]), np.cos(d[:, 2]))
        out.append({
            "noise": g[k].tolist(), "robots": int(m.sum()),
            "anis": a["anis"], "anis_bounds_95": list(a["bounds_95"]), "corrections": a["count"],
            "pose_anees": float(np.nanmean(pose)) if runs else float("nan"),
            "pose_anees_bounds_95": list(cs.chi2_bounds(3, runs)), "pose_runs": runs,
            "landmark_anees": lm_sum / lm_cnt if lm_cnt else float("nan"),
            "landmark_anees_bounds_95": list(cs.chi2_bounds(2, lm_cnt)), "landmark_blocks": lm_cnt,
            "rmse_xytheta": [float(np.sqrt(np.mean(d[:, 0] ** 2))), float(np.sqrt(np.mean(d[:, 1] ** 2))),
                             float(np.sqrt(np.mean(dth ** 2)))],
        })
    for h in (sim, bt):
        h.close()
    return {"world": "dense_world(20)", "groups": K, "robots_per_group": M, "steps": steps, "seed": seed,
            "q_grid": QS, "r_grid": RS, "points": out}


def timing(pkg, torch, n, B, steps, warmup, repeats, traj, seed):
    T = 2 * warmup + 2 * steps * repeats
    tr = pkg.tracegen.simulate_known(world_for(pkg, n), min(traj, B), T, seed=seed)
    reps = -(-B // tr["twists"].shape[1])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (1, reps) + (1,) * (a.ndim - 2))[:, :B])  # noqa: E731
    d = [torch.from_numpy(tile(tr[k])).cuda() for k in ("twists", "xy", "vis")]
    torch.cuda.synchronize()
    bt = pkg.EKFBatch(B, n)
    ref = np.array([1e-4, 1e-4, 1e-4, 0.01, 0.01])
    setting = {False: lambda: bt.set_noise(), True: lambda: bt.set_noise(ref[:3], ref[3:])}
    t = 0
    for on in (False, True):
        setting[on]()
        for _ in range(warmup):
            bt.step_known_dev(*(x[t].data_ptr() for x in d))
            t += 1
    ms = {False: [], True: []}
    for _ in range(repeats):
        for on in (False, True):
            setting[on]()
            bt.sync()
            bt.timer_start()
            for _ in range(steps):
                bt.step_known_dev(*(x[t].data_ptr() for x in d))
                t += 1
            ms[on].append(bt.timer_stop() / steps)
    bt.close()
    del d
    torch.cuda.empty_cache()
    off, on = float(np.median(ms[False])), float(np.median(ms[True]))
    return {"n": n, "B": B, "layout": "tile" if n == 20 else ("staircase" if n <= 64 else "wide"),
            "step_ms_default": round(off, 4), "step_ms_default_min_max": [round(min(ms[False]), 4), round(max(ms[False]), 4)],
            "step_ms_noise": round(on, 4), "step_ms_noise_min_max": [round(min(ms[True]), 4), round(max(ms[True]), 4)],
            "noise_overhead": round(on / off - 1.0, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots-per-point", type=int, default=256)
    ap.add_argument("--steps", type=int, default=140, help="SLAM steps of the sweep")
    ap.add_argument("--time-steps", type=int, default=10, help="timed steps per repeat and kernel")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--traj", type=int, default=1024, help="distinct simulated trajectories of the timing runs")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch

    import ekf_slam_ml_b200 as pkg
    if pkg.device_count() == 0 or not torch.cuda.is_available():
        raise SystemExit("noise_sweep.py needs a CUDA device")
    out = {"bench": "noise_sweep", "gpu": gpu_info(), "sweep": sweep(pkg, a.robots_per_point, a.steps, a.seed),
           "timing": [timing(pkg, torch, n, B, a.time_steps, a.warmup, a.repeats, a.traj, a.seed + 1) for n, B in TIMING]}
    out["gpu_after"] = gpu_info()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
