"""Monte-Carlo accuracy report: the reference README's "Actual / Odom / Slam" comparison
(nuslam/README.md:98-114, one run on one seed) over a whole batch of seeds, entirely on the GPU:
on-device simulator (tube_world restatement) -> batched EKF step, plus a prediction-only batch fed the same twists
(what the motion model alone makes of the 10 Hz odometer twist) and the 100 Hz wheel odometer of the node.
It also scores the filters' consistency: the average NEES (ANEES) of the pose and the landmarks over the batch,
beside the chi-square interval a consistent filter falls in.

    python -m ekf_slam_ml_b200.report --robots 4096 --steps 140 [--nees-every K] [--json]

(`python ekf-slam-ml_b200/report.py ...` works too.)  SURVEY.md §8(f)-4.
"""
import argparse
import json
import os
import sys

import numpy as np


def _rmse(est, truth):
    d = est[:, :2] - truth[:, :2]
    dth = np.arctan2(np.sin(est[:, 2] - truth[:, 2]), np.cos(est[:, 2] - truth[:, 2]))
    return [float(np.sqrt(np.mean(d[:, 0] ** 2))), float(np.sqrt(np.mean(d[:, 1] ** 2))),
            float(np.sqrt(np.mean(dth ** 2)))]


def _anees(cs, stats, key, dof):
    """ANEES of the pose (dof 3) or landmark (dof 2) blocks of an EKFBatch.nees() partial, with its 95 % interval."""
    c = cs.anees_from_stats(stats)
    runs = c[f"{key}_count"]
    return {"anees": c[f"{key}_anees"], "dof": dof, "runs": runs, "singular": c[f"{key}_singular"],
            "bounds_95": list(cs.chi2_bounds(dof, runs))}


def run(pkg, robots=4096, steps=140, seed=0, device=0, world=None, nees_every=0):
    """Returns a dict with the batch statistics after `steps` SLAM steps (11 simulator ticks each; one lap of the
    follow_circle trajectory is about 114 steps).  With nees_every = K > 0 the SLAM batch's pose ANEES is also recorded
    after every K-th step, on the device from the simulator's truth (no host round trip per step)."""
    import torch
    tg = pkg.tracegen
    world = world or tg.dense_world(20)
    n = world.n_slots
    sim = pkg.TubeWorld(world, robots, seed=seed, device=device)
    slam = pkg.EKFBatch(robots, n, device=device)
    blind = pkg.EKFBatch(robots, n, device=device)
    slam.set_nis(True)  # innovation consistency of every correction, on the device
    sim.use_stream(slam.stream)
    p = sim.device_pointers()
    no_vis = torch.zeros(robots * n, dtype=torch.uint8, device=f"cuda:{device}")
    series_at = list(range(nees_every, steps + 1, nees_every)) if nees_every > 0 else []
    series = torch.zeros((len(series_at), 8), dtype=torch.float64, device=f"cuda:{device}")  # one out8 per record
    torch.cuda.synchronize()
    for t in range(1, steps + 1):
        sim.step_known()
        slam.step_known_dev(p["twists"], p["xy"], p["vis"])
        if nees_every > 0 and t % nees_every == 0:
            slam.nees_dev(p["truth"], series[t // nees_every - 1].data_ptr())
        slam.sync()  # the prediction-only batch runs on its own stream: order it after this step's inputs
        blind.step_known_dev(p["twists"], p["xy"], no_vis.data_ptr())
        blind.sync()
    d = sim.download()
    truth, odom = d["truth"], d["odom"]
    est, pred = slam.poses()[:, [1, 2, 0]], blind.poses()[:, [1, 2, 0]]  # (theta, x, y) -> (x, y, theta)
    lm = slam.states()[:, 3:].reshape(robots, n, 2)
    nt = min(world.n_tubes, n)  # every tube's slot is initialised by the first measurement() call (ekf_slam.cpp:113-128)
    tubes = np.stack([world.tubes_x[:nt], world.tubes_y[:nt]], axis=1)[None]
    lm_err = np.linalg.norm(lm[:, :nt] - tubes, axis=2)
    out = {
        "robots": int(robots), "steps": int(steps), "seed": int(seed), "updates": int(slam.update_count),
        "actual_mean_xy": [float(truth[:, 0].mean()), float(truth[:, 1].mean())],
        "rmse_xytheta": {"slam": _rmse(est, truth), "prediction_only": _rmse(pred, truth), "wheel_odometry": _rmse(odom, truth)},
        "worst_xy_error": {"slam": float(np.abs(est[:, :2] - truth[:, :2]).max()),
                           "prediction_only": float(np.abs(pred[:, :2] - truth[:, :2]).max()),
                           "wheel_odometry": float(np.abs(odom[:, :2] - truth[:, :2]).max())},
        "landmark_rmse": float(np.sqrt(np.mean(lm_err ** 2))),
        "landmarks": int(nt),
    }
    # consistency: NEES against the simulator's truth; slots without a tube are not scored
    lm_truth = np.full((n, 2), np.nan)
    lm_truth[:nt] = tubes[0]
    cs = pkg.consistency
    ns, nb = slam.nees(truth, lm_truth)["stats"], blind.nees(truth)["stats"]
    out["consistency"] = {"slam": {"pose": _anees(cs, ns, "pose", 3), "landmarks": _anees(cs, ns, "landmark", 2)},
                          "prediction_only": {"pose": _anees(cs, nb, "pose", 3)}}
    ni = slam.nis()
    out["consistency"]["slam"]["innovations"] = {"anis": ni["anis"], "dof": 2, "bounds_95": list(ni["bounds_95"]),
                                                 "corrections": ni["count"], "nonfinite": ni["nonfinite"]}
    if series_at:
        out["consistency"]["pose_anees_series"] = {
            "steps": series_at, "anees": [cs.anees_from_stats(v)["pose_anees"] for v in series.cpu().numpy()]}
    for h in (sim, slam, blind):
        h.close()
    return out


def markdown(r):
    rows = ["Path type | x RMSE (m) | y RMSE (m) | theta RMSE (rad) | worst |x|,|y| error (m)", "--- | --- | --- | --- | ---"]
    for key, name in (("wheel_odometry", "Odom (100 Hz wheel integration)"), ("prediction_only", "Prediction only (10 Hz twist)"),
                      ("slam", "Slam")):
        e = r["rmse_xytheta"][key]
        rows.append(f"{name} | {e[0]:.5f} | {e[1]:.5f} | {e[2]:.5f} | {r['worst_xy_error'][key]:.5f}")
    head = (f"{r['robots']} robots x {r['steps']} SLAM steps (seed {r['seed']}), {r['updates']} landmark corrections; "
            f"landmark RMSE {r['landmark_rmse']:.5f} m over {r['landmarks']} landmarks per robot")
    text = head + "\n\n" + "\n".join(rows)
    c = r.get("consistency")
    if c:
        rows = ["Consistency | block | dof | ANEES | 95 % interval | runs | singular", "--- | --- | --- | --- | --- | --- | ---"]
        for name, key, block in (("Prediction only", "prediction_only", "pose"), ("Slam", "slam", "pose"),
                                 ("Slam", "slam", "landmarks")):
            e = c[key][block]
            rows.append(f"{name} | {block} | {e['dof']} | {e['anees']:.3f} | {e['bounds_95'][0]:.3f} .. "
                        f"{e['bounds_95'][1]:.3f} | {e['runs']} | {e['singular']}")
        e = c["slam"].get("innovations")
        if e:  # NIS needs no truth: ANIS over every scored correction (columns: ANIS, corrections, non-finite)
            rows.append(f"Slam | innovations | {e['dof']} | {e['anis']:.3f} | {e['bounds_95'][0]:.3f} .. "
                        f"{e['bounds_95'][1]:.3f} | {e['corrections']} | {e['nonfinite']}")
        text += ("\n\nANEES: mean NEES over the runs; a consistent filter lies inside the interval, an overconfident one "
                 "above it.\n\n" + "\n".join(rows))
        if e:
            text += ("\n\nInnovations: ANIS, the mean NIS over every scored correction (needs no truth); its runs column "
                     "counts corrections, its singular column non-finite values.")
        sr = c.get("pose_anees_series")
        if sr:
            text += "\n\nSlam pose ANEES by step: " + ", ".join(f"{t}: {v:.3f}" for t, v in zip(sr["steps"], sr["anees"]))
    return text


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=140)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--nees-every", type=int, default=0, metavar="K",
                    help="also record the SLAM batch's pose ANEES after every K-th step (on the device)")
    ap.add_argument("--json", action="store_true")
    a = ap.parse_args(argv)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import ekf_slam_ml_b200 as pkg
    r = run(pkg, a.robots, a.steps, a.seed, a.device, nees_every=a.nees_every)
    print(json.dumps(r) if a.json else markdown(r))


if __name__ == "__main__":
    main()
