#!/usr/bin/env python
"""Generates tests/golden/*.npz by running the REFERENCE ITSELF (oracle/_ref/libekf_ref.so = the reference's
rigid2d sources compiled unmodified, see oracle/Makefile) on seeded nurtlesim-shaped inputs.

Run with a checkout of the reference:   EKF_SLAM_REFERENCE=<checkout> python scripts/make_golden.py
The fixtures travel with the repo, so the tests need neither the reference nor oracle/_ref.
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _oracle  # noqa: E402
import ekf_slam_ml_b200 as pkg  # noqa: E402  (only its host-side trace generator is used here)

GOLD = os.path.join(ROOT, "tests", "golden")
dp = ctypes.POINTER(ctypes.c_double)
ip = ctypes.POINTER(ctypes.c_int)
u8p = ctypes.POINTER(ctypes.c_uint8)


def main():
    os.makedirs(GOLD, exist_ok=True)
    _oracle.build_oracle()
    L = _oracle.ref_lib()
    assert L is not None, "needs oracle/_ref: set EKF_SLAM_REFERENCE to a checkout of the reference"
    tg = pkg.tracegen
    n = 20
    CK = [0, 1, 2, 5, 20, 59]

    # ---- cfg1: known association, default 10-tube world
    tr = tg.simulate_known(tg.default_world(n), 1, 60, seed=101)
    R = _oracle.RefEKF(n)
    states, sigmas = [], []
    for t in range(60):
        R.prediction(*tr["twists"][t, 0])
        R.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        if t in CK:
            states.append(R.state)
            sigmas.append(R.sigma)
    # Mahalanobis distances of a few probe measurements to every tube at the end of the run
    probes = np.array([[0.3, -0.2], [0.55, 0.1], [-0.4, 0.35], [0.05, 0.62]])
    maha = np.array([[R.maha(px, py, i) for i in range(n)] for px, py in probes])
    np.savez_compressed(os.path.join(GOLD, "ekf_known_n20.npz"), twists=tr["twists"][:, 0], xy=tr["xy"][:, 0],
                        vis=tr["vis"][:, 0], checkpoints=np.array(CK), state=np.array(states), sigma=np.array(sigmas),
                        maha_probes=probes, maha=maha)

    # ---- cfg2 (filter side): unknown association on unlabelled, shuffled readings
    tu = tg.simulate_unknown(tg.default_world(n), 1, 60, seed=202)
    R = _oracle.RefEKF(n)
    O = _oracle.OracleEKF(n)
    kr = np.zeros(n, np.uint8)
    ko = np.zeros(n, np.uint8)
    states, sigmas, known_hist, assoc_hist = [], [], [], []
    for t in range(60):
        R.prediction(*tu["twists"][t, 0])
        O.prediction(*tu["twists"][t, 0])
        m = int(tu["count"][t, 0])
        R.data_association(tu["meas"][t, 0, :m], kr)
        a, dmin, sec, cr = O.data_association(tu["meas"][t, 0, :m], ko)
        assert np.array_equal(kr, ko)
        row = np.full(tu["meas"].shape[2], -9, np.int32)
        row[:m] = a
        assoc_hist.append(row)
        known_hist.append(kr.copy())
        if t in CK:
            states.append(R.state)
            sigmas.append(R.sigma)
    np.savez_compressed(os.path.join(GOLD, "ekf_unknown_n20.npz"), twists=tu["twists"][:, 0], meas=tu["meas"][:, 0],
                        count=tu["count"][:, 0], checkpoints=np.array(CK), state=np.array(states), sigma=np.array(sigmas),
                        known=np.array(known_hist), assoc_from_restatement=np.array(assoc_hist))

    # ---- a mid-sized map (n = 100) to pin the O(N^2) form away from the reference's operating point
    n2 = 100
    w = tg.grid_world(10, 10, pitch=0.35, n_slots=n2, max_visible=0.9)
    t2 = tg.simulate_known(w, 1, 12, seed=303)
    R = _oracle.RefEKF(n2)
    for t in range(12):
        R.prediction(*t2["twists"][t, 0])
        R.measurement(t2["xy"][t, 0], t2["vis"][t, 0])
    np.savez_compressed(os.path.join(GOLD, "ekf_known_n100.npz"), twists=t2["twists"][:, 0], xy=t2["xy"][:, 0],
                        vis=t2["vis"][:, 0], state=R.state, sigma=R.sigma)

    # ---- laser front end: scans -> reference CircleFitting
    ts = tg.simulate_scans(tg.default_world(n), 3, 8, seed=404)
    scans = ts["ranges"].reshape(-1, 360)  # float32 as on the wire
    MAXC = 16
    centers = np.zeros((scans.shape[0], MAXC, 2))
    counts = np.zeros(scans.shape[0], np.int32)
    cl_sizes, cl_cxr, cl_flag = [], [], []
    for s in range(scans.shape[0]):
        r64 = scans[s].astype(np.float64)
        c = np.zeros(2 * MAXC)
        k = L.ref_circles(r64.ctypes.data_as(dp), 360, c.ctypes.data_as(dp), MAXC)
        counts[s] = k
        centers[s] = c.reshape(MAXC, 2)
        sizes = np.zeros(64, np.int32)
        fr = np.zeros(720)
        fxy = np.zeros(1440)
        nc = L.ref_cluster(r64.ctypes.data_as(dp), 360, sizes.ctypes.data_as(ip), 64, fr.ctypes.data_as(dp),
                           fxy.ctypes.data_as(dp), 720)
        cxr = np.zeros(3 * nc)
        fl = np.zeros(nc, np.uint8)
        L.ref_fit_clusters(fxy.ctypes.data_as(dp), sizes.ctypes.data_as(ip), nc, cxr.ctypes.data_as(dp),
                           fl.ctypes.data_as(u8p))
        pad_s = np.zeros(64, np.int32)
        pad_s[:nc] = sizes[:nc]
        pad_c = np.zeros((64, 3))
        pad_c[:nc] = cxr.reshape(nc, 3)
        pad_f = np.zeros(64, np.uint8)
        pad_f[:nc] = fl
        cl_sizes.append(pad_s)
        cl_cxr.append(pad_c)
        cl_flag.append(pad_f)
    np.savez_compressed(os.path.join(GOLD, "circles_scans.npz"), ranges=scans, centers=centers, counts=counts,
                        cluster_sizes=np.array(cl_sizes), cluster_cxr=np.array(cl_cxr), cluster_is_circle=np.array(cl_flag))

    # ---- eigenvalue fallback (circle_fitting.cpp:187-197): clusters in coordinates so large that no eigenvalue of
    # Q lies in (0, 1000); the reference then takes eig_gen's index 0, which LAPACK's dgeev makes the negative one
    rng = np.random.default_rng(20261018)
    fb_clusters, fb_sizes = [], []
    for _ in range(160):
        npts = int(rng.integers(7, 40))
        R = rng.uniform(500, 30000)
        cx, cy = rng.uniform(-5e4, 5e4, 2)
        a0, span = rng.uniform(0, 2 * np.pi), rng.uniform(0.3, 2.5)
        t = a0 + np.linspace(0, span, npts)
        fb_clusters.append(np.stack([cx + R * np.cos(t) + rng.normal(0, 0.05 * R, npts),
                                     cy + R * np.sin(t) + rng.normal(0, 0.05 * R, npts)], 1))
        fb_sizes.append(npts)
    fb_flat = np.ascontiguousarray(np.concatenate(fb_clusters))
    fb_sizes = np.array(fb_sizes, dtype=np.int32)
    fb_cxr = np.zeros((len(fb_sizes), 3))
    fb_isc = np.zeros(len(fb_sizes), np.uint8)
    L.ref_fit_clusters(fb_flat.ctypes.data_as(dp), fb_sizes.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), len(fb_sizes),
                       fb_cxr.ctypes.data_as(dp), fb_isc.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
    np.savez(os.path.join(GOLD, "circles_fallback.npz"), flat_xy=fb_flat, sizes=fb_sizes, cxr=fb_cxr, is_circle=fb_isc)

    # ---- helpers on the path
    rng = np.random.default_rng(5)
    ang = np.concatenate([rng.uniform(-30, 30, 200), [0.0, np.pi, -np.pi, 2 * np.pi, 7.0, -7.0, 100.0]])
    norm = np.array([L.ref_normalize_angle(float(a)) for a in ang])
    wheels = rng.uniform(-0.3, 0.3, (50, 2))
    tw = np.zeros((50, 2))
    for k in range(50):
        o = np.zeros(2)
        L.ref_body_twist(ctypes.c_double(0.16), ctypes.c_double(0.033), ctypes.c_double(wheels[k, 0]),
                         ctypes.c_double(wheels[k, 1]), o.ctypes.data_as(dp))
        tw[k] = o
    np.savez_compressed(os.path.join(GOLD, "helpers.npz"), angles=ang, normalized=norm, wheels=wheels, twists=tw)

    # ---- DiffDrive::updatePose on the seeded cases of tests/test_oracle_cpu.py::test_odometry_restatement_is_pinned
    pose_out = []
    for pose, l, r in _oracle.odometry_inputs():
        b = pose.copy()
        L.ref_update_pose(ctypes.c_double(0.16), ctypes.c_double(0.033), b.ctypes.data_as(dp), ctypes.c_double(l),
                          ctypes.c_double(r))
        pose_out.append(b)
    np.savez_compressed(os.path.join(GOLD, "odometry.npz"), pose_out=np.array(pose_out))
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == "__main__":
    main()
