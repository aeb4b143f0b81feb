"""GPU parity: the CUDA EKF-SLAM path (through the C ABI) against the CPU oracle on identical seeded inputs.

Bar (BASELINE.json north_star): association indices / landmark counts bit-exact away from threshold ties;
state and covariance within 1e-9 in the scaled metric of tests/_oracle.py (sigma_err / state_err)."""
import numpy as np
import pytest

import _single as single
from _batch import tie_margin
from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu

TOL = 1e-9


def _trace(pkg, n_slots, steps, seed, world=None):
    tg = pkg.tracegen
    w = world or (tg.default_world(n_slots) if n_slots >= 10 else None)
    return tg.simulate_known(w, 1, steps, seed=seed)


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_known_association_default_world(gpu_pkg, engine):
    """cfg1: nuslam known association on the default 10-tube world, n = 20 slots."""
    tr = _trace(gpu_pkg, 20, 150, seed=11)
    f = gpu_pkg.EKF_SLAM(20, engine=single.engine(gpu_pkg, engine))
    o = OracleEKF(20)
    ex, es = single.parity_known(f, o, tr, check_every=10)
    assert f.init_flag and o.init_flag
    assert f.update_count == int(tr["vis"].sum())
    assert ex < TOL and es < TOL, (ex, es)


@pytest.mark.parametrize("n,engine", [(3, "fused"), (14, "fused"), (33, "fused"), (64, "fused"), (33, "stream"),
                                      (100, "stream")])
def test_known_association_other_sizes(gpu_pkg, n, engine):
    """Generic-n code paths (the n=20 kernel is a specialised instantiation)."""
    rng = np.random.default_rng(n)
    lm = rng.uniform(-1.5, 1.5, (n, 2))
    f = gpu_pkg.EKF_SLAM(n, engine=single.engine(gpu_pkg, engine))
    o = OracleEKF(n)
    worst = 0.0
    for t in range(25):  # by hand: each step's readings are taken from the oracle's current pose
        dth, dx = 0.05 + rng.normal(0, 0.01), 0.01 + rng.normal(0, 0.002)
        if t % 7 == 3:
            dth = 1e-8  # straight-line branch of the motion model (ekf_slam.cpp:79)
        f.prediction((dth, dx))
        o.prediction(dth, dx)
        th, x, y = o.state[:3]
        rel = lm - [x, y]
        c, s = np.cos(-th), np.sin(-th)
        xy = np.stack([c * rel[:, 0] - s * rel[:, 1], s * rel[:, 0] + c * rel[:, 1]], 1) + rng.normal(0, 0.005, (n, 2))
        vis = (np.hypot(rel[:, 0], rel[:, 1]) < 1.0).astype(np.uint8) if t > 0 else np.zeros(n, np.uint8)
        f.measurement(xy.ravel(), vis)
        o.measurement(xy.ravel(), vis)
        worst = max(worst, state_err(f.state, o.state), sigma_err(f.sigma, o.sigma))
    assert worst < TOL, worst


def _unknown_run(gpu_pkg, n, eng, steps, seed, n_tubes=None):
    tg = gpu_pkg.tracegen
    w = tg.default_world(n)
    if n_tubes:
        w = tg.dense_world(n_tubes)
        w.n_slots = n
    tr = tg.simulate_unknown(w, 1, steps, seed=seed)
    f = gpu_pkg.EKF_SLAM(n, engine=eng)
    o = OracleEKF(n)
    kf = np.zeros(n, np.uint8)
    ko = np.zeros(n, np.uint8)
    worst = 0.0
    n_meas = n_tie = 0
    for t in range(steps):
        res = single.step_unknown(f, tr, t, kf)
        a_o, dmin_o, sec_o, cr_o = single.step_unknown(o, tr, t, ko)
        # a decision is "away from a tie" when neither gate nor the runner-up is within 1e-6 (relative) of dmin
        clear = tie_margin(dmin_o, sec_o) > 1e-6 * np.maximum(1.0, np.abs(dmin_o))
        n_meas += len(a_o)
        n_tie += int((~clear).sum())
        assert np.array_equal(res["assoc"][clear], a_o[clear]), (t, res["assoc"], a_o)
        assert np.array_equal(res["created"][clear], cr_o[clear])
        assert np.array_equal(kf, ko), (t, kf, ko)
        np.testing.assert_allclose(res["dmin"], dmin_o, rtol=1e-7, atol=1e-9)
        worst = max(worst, state_err(f.state, o.state), sigma_err(f.sigma, o.sigma))
    return worst, n_meas, n_tie, int(ko.sum())


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_unknown_association(gpu_pkg, engine):
    """cfg2 filter side: Mahalanobis gating + landmark initialisation, n = 20 slots, 10 tubes."""
    worst, n_meas, n_tie, known = _unknown_run(gpu_pkg, 20, single.engine(gpu_pkg, engine), 120, seed=5)
    assert n_meas > 300 and known >= 5
    assert n_tie == 0
    assert worst < TOL, worst


def test_unknown_association_map_full(gpu_pkg):
    """More tubes (20) than slots (8): once the map is full unmatched measurements are dropped (ekf_slam.cpp:318)."""
    worst, n_meas, n_tie, known = _unknown_run(gpu_pkg, 8, gpu_pkg.ENGINE_FUSED, 60, seed=9, n_tubes=20)
    assert known == 8
    assert worst < TOL, worst


def test_maha_seam_and_getters(gpu_pkg):
    tr = _trace(gpu_pkg, 20, 30, seed=2)
    f = gpu_pkg.EKF_SLAM(20)
    o = OracleEKF(20)
    single.parity_known(f, o, tr, check_every=100)
    for i in (0, 3, 9):
        d_f = f.calculate_maha_dis((0.3, -0.2), i)
        d_o = o.maha(0.3, -0.2, i)
        assert abs(d_f - d_o) <= 1e-9 * max(1.0, abs(d_o))
    s = o.state
    assert abs(f.getStateTheta() - s[0]) < 1e-12 and abs(f.getStateX() - s[1]) < 1e-12
    assert f.getStateLandmark().shape == (40, 1)
    g = f.clone()
    assert np.array_equal(g.state, f.state) and np.array_equal(g.sigma, f.sigma)


def test_pose_read_path_follows_every_way_the_state_can_change(gpu_pkg):
    """The small engine leaves the pose in mapped pinned memory and the facades serve theta / x / y from one read; every
    verb that changes the state - including the ones that do not launch the fused kernel - must be seen by the getters."""
    import ctypes
    tr = _trace(gpu_pkg, 20, 6, seed=8)
    f = gpu_pkg.EKF_SLAM(20)
    o = OracleEKF(20)
    for t in range(3):  # by hand: the getters are read between prediction() and measurement()
        f.prediction(tuple(tr["twists"][t, 0]))
        o.prediction(*tr["twists"][t, 0])
        assert abs(f.getStateTheta() - o.state[0]) < 1e-12 and abs(f.getStateX() - o.state[1]) < 1e-12
        f.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        o.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        assert abs(f.getStateTheta() - o.state[0]) < 1e-11 and abs(f.getStateY() - o.state[2]) < 1e-11
        assert np.allclose(f.state[:3], [f.getStateTheta(), f.getStateX(), f.getStateY()], rtol=0, atol=0)
    s = f.state
    s[:3] = [0.25, -1.5, 2.75]
    f.state = s                                    # set_state: a plain copy, no kernel
    assert (f.getStateTheta(), f.getStateX(), f.getStateY()) == (0.25, -1.5, 2.75)
    f.prediction((0.0, 0.0))                       # back on the kernel path
    assert f.getStateX() == f.state[1] and f.getStateTheta() == f.state[0]
    g = f.clone()
    assert g.getStateX() == f.getStateX() and g.getStateY() == f.getStateY()
    # a caller that took the device pointers may write the state behind the handle: the getter must read the device
    L = gpu_pkg._lib.load()
    st = ctypes.c_void_p()
    assert L.ekf_device_pointers(f._h, None, None, ctypes.byref(st)) == 0 and st.value
    import torch

    class _View:  # three doubles at the state pointer, as a CUDA array
        __cuda_array_interface__ = {"shape": (3,), "typestr": "<f8", "data": (st.value, False), "version": 2}
    torch.as_tensor(_View(), device="cuda").copy_(torch.tensor([1.0, 2.0, 3.0], dtype=torch.float64))
    torch.cuda.synchronize()
    f._pose_cache = None  # the Python facade caches per verb; the write above went around it
    assert (f.getStateTheta(), f.getStateX(), f.getStateY()) == (1.0, 2.0, 3.0)


def test_deferred_prediction_is_invisible(gpu_pkg):
    """On the small engine prediction() only records the twist; it is applied by the next measurement() /
    data_association() kernel or by whatever verb looks at the filter first.  No call order may see the difference."""
    tr = _trace(gpu_pkg, 20, 8, seed=12)
    f = gpu_pkg.EKF_SLAM(20)
    o = OracleEKF(20)
    tw = [tuple(tr["twists"][t, 0]) for t in range(8)]
    # two predictions in a row, then a getter
    for t in (0, 1):
        f.prediction(tw[t])
        o.prediction(*tw[t])
    assert state_err(f.state, o.state) < TOL
    # prediction, then verbs that read Sigma / distances / copies
    f.measurement(tr["xy"][2, 0], tr["vis"][2, 0])
    o.measurement(tr["xy"][2, 0], tr["vis"][2, 0])
    f.prediction(tw[3])
    o.prediction(*tw[3])
    assert abs(f.calculate_maha_dis((0.3, -0.2), 1) - o.maha(0.3, -0.2, 1)) <= 1e-9 * max(1.0, abs(o.maha(0.3, -0.2, 1)))
    f.prediction(tw[4])
    o.prediction(*tw[4])
    g = f.clone()
    assert sigma_err(g.sigma, o.sigma) < TOL and state_err(g.state, o.state) < TOL
    assert np.array_equal(g.sigma, f.sigma) and np.array_equal(g.state, f.state)
    # prediction, an EMPTY association call (nothing to launch), then the measurement that carries it
    known = np.ones(20, np.uint8)
    f.prediction(tw[5])
    o.prediction(*tw[5])
    f.data_association(np.zeros((0, 2)), known)
    f.measurement(tr["xy"][6, 0], tr["vis"][6, 0])
    o.measurement(tr["xy"][6, 0], tr["vis"][6, 0])
    assert sigma_err(f.sigma, o.sigma) < TOL and state_err(f.state, o.state) < TOL
    # prediction, then a state overwrite: the prediction comes first, the overwrite wins
    f.prediction(tw[7])
    o.prediction(*tw[7])
    s0 = o.state.copy()
    s0[:3] = [0.1, 0.2, 0.3]
    f.state = s0
    assert np.array_equal(f.state, s0) and sigma_err(f.sigma, o.sigma) < TOL


def test_normalize_angle_device_twin_is_bit_exact(gpu_pkg):
    """rigid2d::normalize_angle: the device twin must equal the C library fmod formulation bit for bit."""
    import ctypes
    from _oracle import oracle_lib
    L = oracle_lib()
    rng = np.random.default_rng(0)
    vals = np.concatenate([rng.uniform(-40, 40, 20000), rng.uniform(-7, 7, 20000),
                           np.array([0.0, -0.0, np.pi, -np.pi, 2 * np.pi, -2 * np.pi, 3 * np.pi, 1e-300, 6.283185307179586,
                                     6.2831853071795862, 12.566370614359172, 1e5, -1e5, 1e7, -3e9]),
                           np.nextafter(np.pi * np.arange(-8, 9), np.inf), np.nextafter(np.pi * np.arange(-8, 9), -np.inf)])
    got = gpu_pkg.normalize_angle(vals)
    want = np.array([L.oracle_normalize_angle(float(v)) for v in vals])
    assert np.array_equal(single.bits(got), single.bits(want))
    # golden values of rigid2d/tests/tests.cpp:322-331
    g = gpu_pkg.normalize_angle(np.deg2rad([30.0, 230.0, -330.0]))
    np.testing.assert_allclose(g, [0.523599, -2.26893, 0.523599], rtol=1.2e-5)


def test_update_pose_device_twin(gpu_pkg):
    """DiffDrive::updatePose on the device vs the pinned C restatement (CUDA sincos / acos / asin differ from libm in
    the last bits, and acos amplifies them for small rotations: 1e-9 absolute) + the reference's known answers."""
    import ctypes
    from _oracle import oracle_lib
    L = oracle_lib()
    d, P = ctypes.c_double, ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(9)
    n = 5000
    poses = np.column_stack([rng.normal(size=n), rng.normal(size=n), rng.uniform(-7, 7, size=n)])
    left, right = rng.uniform(-0.2, 0.2, size=n), rng.uniform(-0.2, 0.2, size=n)
    left[::3], right[::3] = rng.uniform(-40, 40, size=len(left[::3])), rng.uniform(-40, 40, size=len(left[::3]))
    right[::7] = left[::7] + rng.uniform(-1e-6, 1e-6, size=len(left[::7]))
    got = gpu_pkg.update_pose(0.16, 0.033, poses, left, right)
    want = poses.copy()
    for k in range(n):
        L.oracle_update_pose(d(0.16), d(0.033), want[k].ctypes.data_as(P), d(left[k]), d(right[k]))
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-9)
    # rigid2d/tests/tests.cpp:334-383
    dd = gpu_pkg.DiffDrive(0.2, 0.01)
    dd.updatePose(0.5, 0.5)
    assert abs(dd.getPosition().x - 0.005) < 1e-7 and abs(dd.getPosition().y) < 1e-12
    dd = gpu_pkg.DiffDrive(0.2, 0.01)
    dd.updatePose(-15.7, 15.7)
    assert abs(dd.getTheta() - 1.57) < 2e-5 and abs(dd.getPosition().x) < 1e-12
    dd = gpu_pkg.DiffDrive(0.2, 0.05)
    dd.updatePose(0.0, 2 * 3.1415926)
    assert abs(dd.getTheta() - 1.5708) < 2e-5 and abs(dd.getPosition().x - 0.1) < 2e-6 and abs(dd.getPosition().y - 0.1) < 2e-6


def test_batch_matches_per_filter_oracle(gpu_pkg):
    """cfg3 in miniature: every filter of a batch equals its own oracle run (known association)."""
    tg = gpu_pkg.tracegen
    B, T = 96, 24
    tr = tg.simulate_known(tg.dense_world(20), B, T, seed=3)
    bt = gpu_pkg.EKFBatch(B, 20)
    for t in range(T):
        bt.step_known(np.ascontiguousarray(tr["twists"][t]), np.ascontiguousarray(tr["xy"][t]),
                      np.ascontiguousarray(tr["vis"][t]))
        bt.sync()
    states = bt.states()
    assert bt.update_count == int(tr["vis"].sum())
    worst = 0.0
    for b in range(0, B, 5):
        o = single.run_known(OracleEKF(20), tr, b)
        worst = max(worst, state_err(states[b], o.state), sigma_err(bt.sigma(b), o.sigma))
    assert worst < TOL, worst
    poses = bt.poses()
    assert np.array_equal(poses, states[:, :3])
    err = bt.pose_error(tr["truth"][-1])
    assert err[3] == B and np.all(err[:3] / B < 0.05 ** 2)


@pytest.mark.parametrize("n", [20, 40])
def test_batch_marker_list_equals_dense_arrays(gpu_pkg, n):
    """The fake_sensor marker list (visible markers only, CSR) gives bit-identical filters to the dense arrays the
    SLAM node unpacks it into (nuslam/src/slam.cpp:232-262), including the first call that initialises every slot."""
    tg = gpu_pkg.tracegen
    B, T = 200, 10
    tr = tg.simulate_known(tg.grid_world(8, 5, pitch=0.35) if n != 20 else tg.dense_world(20), B, T, seed=11)
    dense, sparse = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    for t in range(T):
        tw = np.ascontiguousarray(tr["twists"][t])
        xy = np.ascontiguousarray(tr["xy"][t]) * tr["vis"][t].repeat(2, axis=1)  # unlisted slots read (0, 0)
        vis = np.ascontiguousarray(tr["vis"][t])
        dense.step_known(tw, xy, vis)
        off, ids, pts = gpu_pkg.marker_list(xy, vis)
        assert off[-1] == vis.sum() and len(ids) == off[-1]
        sparse.step_known_sparse(tw, off, ids, pts)
        dense.sync()
        sparse.sync()
    assert sparse.update_count == dense.update_count == int(tr["vis"].sum())
    assert np.array_equal(sparse.states(), dense.states())
    for b in (0, B // 2, B - 1):
        assert np.array_equal(sparse.sigma(b), dense.sigma(b))
    # malformed offsets (beyond the list, decreasing) give those filters an empty list instead of a wild read
    bad = gpu_pkg.EKFBatch(B, n)
    ref2 = gpu_pkg.EKFBatch(B, n)
    off, ids, pts = gpu_pkg.marker_list(xy, vis)
    broken = off.copy()
    broken[3] = off[-1] + 1000       # filter 2 ends (and filter 3 starts) outside the list
    tw0 = np.ascontiguousarray(tr["twists"][1])
    bad.step_known_sparse(tw0, broken, ids, pts, total=int(off[-1]))
    ref2.step_known_sparse(tw0, off, ids, pts)
    bad.sync(), ref2.sync()
    sb, sr = bad.states(), ref2.states()
    assert np.all(np.isfinite(sb)) and np.array_equal(sb[4:], sr[4:]) and np.array_equal(sb[:2], sr[:2])
    # an empty list is a prediction-only step
    before = sparse.states()
    sparse.step_known_sparse(np.zeros((B, 2)), np.zeros(B + 1, np.int32), np.zeros(0, np.uint8), np.zeros((0, 2)))
    sparse.sync()
    assert np.array_equal(sparse.states(), before)


def test_batch_checkpoint_resume_is_bit_identical(gpu_pkg, tmp_path):
    """Checkpoint / resume (SURVEY.md §5): a restored batch continues exactly where the original would have."""
    tg = gpu_pkg.tracegen
    B, T, M = 64, 16, 8
    tr = tg.simulate_known(tg.dense_world(20), B, T, seed=21)
    tu = tg.simulate_unknown(tg.default_world(20), B, T, seed=22, m_max=M)
    for mode in ("known", "unknown"):
        a, b = gpu_pkg.EKFBatch(B, 20), gpu_pkg.EKFBatch(B, 20)

        def step(bt, t):
            if mode == "known":
                bt.step_known(np.ascontiguousarray(tr["twists"][t]), np.ascontiguousarray(tr["xy"][t]),
                              np.ascontiguousarray(tr["vis"][t]))
            else:
                bt.step_unknown(np.ascontiguousarray(tu["twists"][t]), np.ascontiguousarray(tu["meas"][t]),
                                np.ascontiguousarray(tu["count"][t]), M)
            bt.sync()

        for t in range(T // 2):
            step(a, t)
        path = str(tmp_path / f"ck_{mode}.npz")
        a.save_checkpoint(path)
        b.load_checkpoint(path)
        assert b.update_count == a.update_count
        for t in range(T // 2, T):
            step(a, t)
            step(b, t)
        assert np.array_equal(a.states(), b.states()) and np.array_equal(a.known, b.known)
        assert np.array_equal(a.sigma(B - 1), b.sigma(B - 1)) and a.update_count == b.update_count
    with pytest.raises(ValueError):
        gpu_pkg.EKFBatch(B + 1, 20).restore(a.checkpoint())


def test_batch_unknown_matches_oracle(gpu_pkg):
    tg = gpu_pkg.tracegen
    B, T, M = 40, 30, 10
    tr = tg.simulate_unknown(tg.default_world(20), B, T, seed=4, m_max=M)
    bt = gpu_pkg.EKFBatch(B, 20)
    assoc = []
    for t in range(T):
        assoc.append(bt.step_unknown(np.ascontiguousarray(tr["twists"][t]), np.ascontiguousarray(tr["meas"][t]),
                                     np.ascontiguousarray(tr["count"][t]), M, want_assoc=True))
    states, known = bt.states(), bt.known
    worst = 0.0
    for b in range(0, B, 3):
        o = OracleEKF(20)
        k = np.zeros(20, np.uint8)
        for t, (a, _, _, _) in enumerate(single.run_unknown(o, tr, k, b)):
            assert np.array_equal(assoc[t][b, :len(a)], a)
            assert np.all(assoc[t][b, len(a):] == -1)
        assert np.array_equal(known[b], k)
        worst = max(worst, state_err(states[b], o.state), sigma_err(bt.sigma(b), o.sigma))
    assert worst < TOL, worst


def test_large_map_stream_engine(gpu_pkg):
    """n = 1,000 landmarks (N = 2,003): the HBM-streamed engine against the O(N^2) oracle, both verbs."""
    n = 1000
    tg = gpu_pkg.tracegen
    w = tg.grid_world(40, 25, pitch=0.45, n_slots=n, max_visible=1.0)
    tr = tg.simulate_known(w, 1, 12, seed=1)
    f = gpu_pkg.EKF_SLAM(n)
    assert f.engine == gpu_pkg.ENGINE_STREAM
    o = OracleEKF(n)
    ex, es = single.parity_known(f, o, tr, check_every=4)
    assert int(tr["vis"].sum()) > 40
    assert ex < TOL and es < TOL, (ex, es)
    # then unknown association on top of the converged map: all landmarks known
    known_f = np.ones(n, np.uint8)
    known_o = np.ones(n, np.uint8)
    tu = tg.simulate_unknown(w, 1, 3, seed=1)
    for t in range(3):  # by hand: association only, no prediction in between
        m = int(tu["count"][t, 0])
        meas = tu["meas"][t, 0, :m]
        # measurements come from a different trajectory prefix, so most will be gated out: both sides must agree
        r = f.data_association(meas, known_f)
        a, dmin, sec, cr = o.data_association(meas, known_o)
        assert np.array_equal(r["assoc"], a)
        np.testing.assert_allclose(r["dmin"], dmin, rtol=1e-7, atol=1e-9)
    assert state_err(f.state, o.state) < TOL and sigma_err(f.sigma, o.sigma) < TOL


def test_large_map_cfg4_size(gpu_pkg):
    """BASELINE cfg4 at its full size (n = 8,192, N = 16,387, Sigma 2.1 GB): 14 corrections through the multi-factor
    DMMA sweep against the O(N^2) oracle, state and the whole covariance."""
    n = 8192
    tg = gpu_pkg.tracegen
    w = tg.grid_world(128, 64, pitch=0.5, n_slots=n, max_visible=0.7)
    tr = tg.simulate_known(w, 1, 6, seed=99)
    f = gpu_pkg.EKF_SLAM(n)
    o = OracleEKF(n)
    done = t = 0
    while done < 10:
        single.step_known(f, tr, t)
        single.step_known(o, tr, t)
        done += int(tr["vis"][t, 0].sum()) if t else 0
        t += 1
    assert f.sweep_count <= 1  # the corrections went through (at most) one sweep so far, the rest is pending
    assert state_err(f.state, o.state) < TOL
    sig, ref = f.sigma, o.sigma
    d = np.sqrt(np.abs(np.diag(ref)))
    worst = 0.0
    for i0 in range(0, ref.shape[0], 256):
        sl = slice(i0, i0 + 256)
        scale = np.maximum(np.maximum(np.abs(ref[sl]), d[sl, None] * d[None, :]), 1e-300)
        worst = max(worst, float(np.max(np.abs(sig[sl] - ref[sl]) / scale)))
    assert worst < TOL, worst
    # the rows / diagonal accessors used by the parity checks of maps too large to read back whole
    rows = np.array([0, 2, 3, 4097, 16386], dtype=np.int64)
    assert np.array_equal(f.sigma_rows(rows), sig[rows]) and np.array_equal(f.sigma_diag, np.diag(sig))


def test_update_count_with_one_sweep_per_correction(gpu_pkg):
    """max_pending = 1 (the reference's schedule): data_association() on the streamed engine must count exactly the
    corrections it applied and must not sweep for a dropped measurement."""
    n = 300
    tg = gpu_pkg.tracegen
    w = tg.grid_world(20, 15, pitch=0.45, n_slots=n, max_visible=1.0)
    tr = tg.simulate_known(w, 1, 3, seed=2)
    f = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
    f.set_max_pending(1)
    o = OracleEKF(n)
    for obj in (f, o):
        single.step_known(obj, tr, 0)
    ids = np.flatnonzero(tr["vis"][1, 0])[:4]
    xy = tr["xy"][1, 0].reshape(-1, 2)[ids]
    meas = np.concatenate([xy, [[55.0, 55.0]]])  # the last one is far from everything: gated out, no correction
    kf, ko = np.ones(n, np.uint8), np.ones(n, np.uint8)
    u0, s0 = f.update_count, f.sweep_count
    r = f.data_association(meas, kf)
    a, _, _, _ = o.data_association(meas, ko)
    applied = int(np.sum(a >= 0))
    assert np.array_equal(r["assoc"], a) and applied >= 3 and a[-1] == -1
    assert f.update_count - u0 == applied
    assert state_err(f.state, o.state) < TOL and sigma_err(f.sigma, o.sigma) < TOL


def test_streamed_filter_on_a_second_device(gpu_pkg):
    """The multi-factor sweep opts in to > 48 KB of shared memory per DEVICE: a filter on device 1 after one on device 0."""
    if gpu_pkg.device_count() < 2:
        pytest.skip("needs two GPUs")
    n = 300
    tg = gpu_pkg.tracegen
    w = tg.grid_world(20, 15, pitch=0.45, n_slots=n, max_visible=1.0)
    tr = tg.simulate_known(w, 1, 4, seed=3)
    for dev in (0, 1):
        f = gpu_pkg.EKF_SLAM(n, device=dev, engine=gpu_pkg.ENGINE_STREAM)
        o = OracleEKF(n)
        ex, es = single.parity_known(f, o, tr, check_every=2)
        assert ex < TOL and es < TOL, (dev, ex, es)


def test_association_log(gpu_pkg, tmp_path):
    """The per-call association record the reference only prints: one CSV line per measurement."""
    tg = gpu_pkg.tracegen
    tu = tg.simulate_unknown(tg.default_world(20), 1, 12, seed=4)
    f = gpu_pkg.EKF_SLAM(20)
    o = OracleEKF(20)
    log = tmp_path / "assoc.csv"
    f.association_log(log)
    kf, ko = np.zeros(20, np.uint8), np.zeros(20, np.uint8)
    expect = []
    for t in range(12):  # by hand: no data_association() call for a step without readings
        m = int(tu["count"][t, 0])
        f.prediction(tuple(tu["twists"][t, 0]))
        o.prediction(*tu["twists"][t, 0])
        if m:
            f.data_association(tu["meas"][t, 0, :m], kf)
            a, dmin, sec, cr = o.data_association(tu["meas"][t, 0, :m], ko)
            expect += [(j, int(a[j]), float(dmin[j]), int(cr[j])) for j in range(m)]
    f.association_log(None)
    rows = np.genfromtxt(log, delimiter=",", names=True)
    assert len(rows) == len(expect) > 20
    assert [int(v) for v in rows["index"]] == [e[0] for e in expect]
    assert [int(v) for v in rows["landmark"]] == [e[1] for e in expect]
    assert [int(v) for v in rows["created"]] == [e[3] for e in expect]
    np.testing.assert_allclose(rows["min_distance"], [e[2] for e in expect], rtol=1e-7, atol=1e-9)


def test_batch_wrappers_reject_wrong_buffers(gpu_pkg):
    bt = gpu_pkg.EKFBatch(8, 20)
    tw = np.zeros((8, 2))
    with pytest.raises(TypeError):
        bt.step_known(tw, np.zeros((8, 40)), np.zeros((8, 20), np.int64))  # visible must be uint8
    with pytest.raises(ValueError):
        bt.step_known(tw, np.zeros((8, 20)), np.zeros((8, 20), np.uint8))  # xy too short
    with pytest.raises(ValueError):
        bt.step_known_sparse(tw, np.zeros(9, np.int32), np.zeros(0, np.uint8), np.zeros((0, 2)), total=5)
    bt.close()


def test_invalid_arguments_do_not_crash(gpu_pkg):
    with pytest.raises(gpu_pkg.EkfError):
        gpu_pkg.EKF_SLAM(0)
    with pytest.raises(gpu_pkg.EkfError):
        gpu_pkg.EKF_SLAM(20, device=99)
    with pytest.raises(gpu_pkg.EkfError):
        gpu_pkg.EKF_SLAM(200, engine=gpu_pkg.ENGINE_FUSED)
    f = gpu_pkg.EKF_SLAM(20)
    with pytest.raises(ValueError):
        f.measurement(np.zeros(10), np.zeros(20, np.uint8))
    known = np.zeros(20, np.uint8)
    f.data_association(np.zeros((0, 2)), known)  # empty measurement list is a no-op
    assert known.sum() == 0 and f.update_count == 0


# ---------------------------------------------------------------- golden vectors from the reference's own source
import os as _os

_GOLD = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_golden_known_association(gpu_pkg, engine):
    """tests/golden/ekf_known_n20.npz: state / Sigma checkpoints and Mahalanobis probes produced by the reference."""
    g = np.load(_os.path.join(_GOLD, "ekf_known_n20.npz"))
    f = gpu_pkg.EKF_SLAM(20, engine=single.engine(gpu_pkg, engine))
    ck = list(g["checkpoints"])
    worst = 0.0
    for t in range(g["twists"].shape[0]):  # by hand: the golden arrays have no trajectory axis
        f.prediction(tuple(g["twists"][t]))
        f.measurement(g["xy"][t], g["vis"][t])
        if t in ck:
            k = ck.index(t)
            worst = max(worst, state_err(f.state, g["state"][k]), sigma_err(f.sigma, g["sigma"][k]))
    assert worst < TOL, worst
    for p, (px, py) in enumerate(g["maha_probes"]):
        for i in range(20):
            want = g["maha"][p, i]
            assert abs(f.calculate_maha_dis((px, py), i) - want) <= 1e-8 * max(1.0, abs(want))


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_golden_unknown_association(gpu_pkg, engine):
    """tests/golden/ekf_unknown_n20.npz: the reference's known_list after every call, state / Sigma checkpoints.

    What comes from where: `known`, `state`, `sigma` were produced by the REFERENCE build (oracle/_ref).  The reference
    exposes no per-measurement association index (it only prints), so `assoc_from_restatement` was produced by
    oracle/ekf_oracle.c on the same run; the reference-owned checkpoints of state and Sigma are what close the loop on
    those indices (a different association would move them far beyond the tolerance)."""
    g = np.load(_os.path.join(_GOLD, "ekf_unknown_n20.npz"))
    f = gpu_pkg.EKF_SLAM(20, engine=single.engine(gpu_pkg, engine))
    known = np.zeros(20, np.uint8)
    ck = list(g["checkpoints"])
    worst = 0.0
    for t in range(g["twists"].shape[0]):  # by hand: the golden arrays have no trajectory axis
        f.prediction(tuple(g["twists"][t]))
        m = int(g["count"][t])
        r = f.data_association(g["meas"][t, :m], known)
        assert np.array_equal(known, g["known"][t])
        assert np.array_equal(r["assoc"], g["assoc_from_restatement"][t, :m])
        if t in ck:
            k = ck.index(t)
            worst = max(worst, state_err(f.state, g["state"][k]), sigma_err(f.sigma, g["sigma"][k]))
    assert worst < TOL, worst


def test_golden_n100(gpu_pkg):
    g = np.load(_os.path.join(_GOLD, "ekf_known_n100.npz"))
    f = gpu_pkg.EKF_SLAM(100)
    for t in range(g["twists"].shape[0]):  # by hand: the golden arrays have no trajectory axis
        f.prediction(tuple(g["twists"][t]))
        f.measurement(g["xy"][t], g["vis"][t])
    assert state_err(f.state, g["state"]) < TOL and sigma_err(f.sigma, g["sigma"]) < TOL


def test_scan_to_map_pipeline(gpu_pkg):
    """cfg2 end to end on the GPU: 360-beam scans -> clustering + circle fit -> data_association, against the same
    pipeline built from the oracles (numpy/LAPACK circle fit feeding the plain-C filter)."""
    import sys
    sys.path.insert(0, _os.path.join(_os.path.dirname(_GOLD), "..", "oracle"))
    import circle_oracle as co
    tg = gpu_pkg.tracegen
    T = 40
    s = tg.simulate_scans(tg.default_world(20), 1, T, seed=8)
    cf = gpu_pkg.CircleFitting()
    f = gpu_pkg.EKF_SLAM(20)
    o = OracleEKF(20)
    kf, ko = np.zeros(20, np.uint8), np.zeros(20, np.uint8)
    n_meas = 0
    for t in range(T):  # by hand: the readings are the circle fit's, not the trace's
        centers, counts = cf.run_batch(s["ranges"][t])
        k = int(counts[0])
        c_o, _ = co.approx_circle_positions(s["ranges"][t, 0].astype(np.float64))
        assert k == len(c_o)
        np.testing.assert_allclose(centers[0, :k], c_o, atol=1e-9)
        f.prediction(tuple(s["twists"][t, 0]))
        o.prediction(*s["twists"][t, 0])
        if k:
            r = f.data_association(centers[0, :k], kf)
            a, dmin, sec, cr = o.data_association(c_o, ko)
            assert np.all(tie_margin(dmin, sec) > 1e-6), "threshold tie in the fixture: pick another seed"
            assert np.array_equal(r["assoc"], a) and np.array_equal(kf, ko)
            n_meas += k
    assert n_meas > 100 and ko.sum() >= 5
    assert state_err(f.state, o.state) < 1e-8 and sigma_err(f.sigma, o.sigma) < 1e-8


def test_delayed_application_is_bit_identical(gpu_pkg):
    """Accumulating up to 20 corrections per pass over Sigma (ekf_large_delayed.cuh) must give exactly the bits of
    the reference's schedule (one pass per correction): every element sees the same FMA sequence."""
    n = 300
    tg = gpu_pkg.tracegen
    w = tg.grid_world(20, 15, pitch=0.4, n_slots=n, max_visible=1.2)
    tr = tg.simulate_known(w, 1, 8, seed=21)
    outs = []
    ks = (1, 2, 3, 8, 14, 15, 20)  # 1..2: register sweep; 3..20: DMMA sweep, 512-column tiles to 14, 256 from 15
    for k in ks:
        f = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
        f.set_max_pending(k)
        f.set_carry_pending(False)  # groups end with the measurement() call
        single.run_known(f, tr)
        outs.append((f.state, f.sigma, f.launch_count))
    assert int(tr["vis"][1:].sum(axis=2).max()) > 15  # some steps need more than one group at k = 8 and fill a group of 15+
    for st, sg, _ in outs[1:]:
        assert np.array_equal(single.bits(st), single.bits(outs[0][0]))
        assert np.array_equal(single.bits(sg), single.bits(outs[0][1]))
    assert outs[ks.index(20)][2] < outs[ks.index(8)][2] < outs[0][2]  # fewer launches: fewer sweeps


def test_pending_factors_carried_across_prediction(gpu_pkg):
    """Default schedule of the streamed engine: factors stay pending across prediction() (mapped through the motion
    Jacobian) and measurement() calls, so sweeps always carry max_pending corrections.  Same filter to rounding as
    the per-call schedule and as the oracle; getters settle the pending factors."""
    n = 300
    tg = gpu_pkg.tracegen
    w = tg.grid_world(20, 15, pitch=0.4, n_slots=n, max_visible=0.55)  # 4-6 visible landmarks per step
    T = 14
    tr = tg.simulate_known(w, 1, T, seed=23)
    a = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
    b = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
    b.set_carry_pending(False)
    o = OracleEKF(n)
    for t in range(T):  # by hand: a getter is read in the middle of the run
        for f in (a, b, o):
            single.step_known(f, tr, t)
        if t == T // 2:  # a getter in the middle settles the factors without changing the outcome
            assert sigma_err(a.sigma, o.sigma) < TOL
    assert a.sweep_count < b.sweep_count             # fewer passes over Sigma
    assert a.update_count == b.update_count == int(tr["vis"].sum())
    assert state_err(a.state, b.state) < 1e-12 and sigma_err(a.sigma, b.sigma) < 1e-11
    assert state_err(a.state, o.state) < TOL and sigma_err(a.sigma, o.sigma) < TOL
