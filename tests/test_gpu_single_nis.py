"""NIS (normalised innovation squared) of the single filter: EKF_SLAM.set_nis / nis / last_nis on the fused engine
(n <= 64: the n = 20 kernel and the generic one) and on the streamed engine.

The NIS variants of the fused kernel and of the streamed engine's gain kernels must leave the filter bit-identical and
add no launch; their accumulators and per-call values follow the numpy restatement of the CPU oracle
(tests/_noise_ref.py), with the scoring rule of the batch engines; a streamed filter with carry_pending off must give
the accumulators of the same filter in a wide batch, bit for bit."""
import numpy as np
import pytest

import _single as single
from _batch import known_trace, robot_frame, run_known
from _noise_ref import DEFAULT_NOISE, NoiseOracle

pytestmark = pytest.mark.gpu

M_MAX = 40
NIS_RTOL = 1e-8  # against the numpy reference; observed deviations are printed
# a noise row of tests/test_gpu_noise.py's grid, so that the NOISE x NIS variants run
NOISE_ROW = np.array([4e-4, 2e-4, 3e-4, 0.003, 0.002])
# (engine, n): the fused n = 20 kernel, the fused generic kernel (NL = 0), the streamed engine at both sizes
FILTERS = [("fused", 20), ("fused", 33), ("stream", 20), ("stream", 100)]


def _make(pkg, engine, n, noise=None):
    f = pkg.EKF_SLAM(n, engine=single.engine(pkg, engine))
    if noise is not None:
        f.set_noise(noise[:3], noise[3:])
    return f


def _nis_dev(got, want, what):
    """Worst relative deviation of the scored entries; the -1 entries must sit exactly where the oracle's do."""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert np.array_equal(got == -1.0, want == -1.0), (what, got, want)
    m = want != -1.0
    if not m.any():
        return 0.0
    return float((np.abs(got[m] - want[m]) / np.maximum(np.abs(want[m]), 1e-300)).max())


# ---------------------------------------------------------------- 1. the NIS variants do not change the filter
@pytest.mark.parametrize("noise", ["reference", "grid"])
@pytest.mark.parametrize("engine,n", FILTERS, ids=[f"{e}-{n}" for e, n in FILTERS])
def test_nis_leaves_filter_unchanged(gpu_pkg, engine, n, noise):
    T = 6
    row = NOISE_ROW if noise == "grid" else None
    tk, tu = single.traces(gpu_pkg, n, T, seed=10 + n, m_max=M_MAX)
    plain, scored = _make(gpu_pkg, engine, n, row), _make(gpu_pkg, engine, n, row)
    scored.set_nis(True)
    kp, ks = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for t in range(T):
        for f in (plain, scored):
            single.step_known(f, tk, t)
        a, b = single.step_unknown(plain, tu, t, kp), single.step_unknown(scored, tu, t, ks)
        for key in ("assoc", "created"):
            assert np.array_equal(a[key], b[key]), (t, key)
        for key in ("dmin", "second"):
            assert np.array_equal(single.bits(a[key]), single.bits(b[key])), (t, key)
        assert np.array_equal(kp, ks), t
    assert np.array_equal(single.bits(plain.state), single.bits(scored.state))
    assert np.array_equal(single.bits(plain.sigma), single.bits(scored.sigma))
    assert plain.update_count == scored.update_count
    assert plain.launch_count == scored.launch_count
    r = scored.nis()
    assert r["count"] > 0 and r["nonfinite"] == 0


# ---------------------------------------------------------------- 2. parity with the numpy reference
@pytest.mark.parametrize("noise", ["reference", "grid"])
@pytest.mark.parametrize("mode", ["known", "unknown"])
@pytest.mark.parametrize("engine,n", FILTERS, ids=[f"{e}-{n}" for e, n in FILTERS])
def test_nis_matches_reference(gpu_pkg, engine, n, mode, noise):
    T = 8
    row = NOISE_ROW if noise == "grid" else np.array(DEFAULT_NOISE)
    tk, tu = single.traces(gpu_pkg, n, T, seed=100 + n, m_max=M_MAX)
    f, o = _make(gpu_pkg, engine, n, row), NoiseOracle(n, row)
    f.set_nis(True)
    worst = 0.0
    kf, ko = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for t in range(T):
        if mode == "known":
            single.step_known(f, tk, t)
            want = single.nis_step_known(o, tk, t)
        else:
            got = single.step_unknown(f, tu, t, kf)
            a, _, want = single.nis_step_unknown(o, tu, t, ko)
            assert np.array_equal(got["assoc"], a), t
        worst = max(worst, _nis_dev(f.last_nis(), want, f"{engine} n={n} {mode} call {t}"))
    r = f.nis()
    assert r["count"] == o.acc[2] and r["nonfinite"] == 0
    for k in (0, 1):
        worst = max(worst, abs(r["stats"][k] - o.acc[k]) / abs(o.acc[k]))
    print(f"{engine} n={n} {mode} {noise}: NIS vs numpy reference, worst relative deviation {worst:.2e}, "
          f"scored {int(o.acc[2])}")
    assert o.acc[2] > 0 and worst < NIS_RTOL


# ---------------------------------------------------------------- 3. streamed equals wide
@pytest.mark.parametrize("carry", [False, True])
def test_streamed_equals_wide(gpu_pkg, carry):
    B, T, n, b = 3, 5, 100, 1
    tr = known_trace(gpu_pkg, n, B, T, seed=700)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_nis(True)
    run_known(gpu_pkg, bt, tr)
    f = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
    f.set_carry_pending(carry)
    f.set_nis(True)
    single.run_known(f, tr, b)
    want = bt.nis(per_filter=True)
    want = np.array([want["nis_sum"][b], want["nis_sq_sum"][b], want["nis_count"][b], want["nis_nonfinite"][b]])
    got = f.nis()["stats"]
    assert got[2] > 0
    if carry:
        assert got[2] == want[2] and got[3] == want[3]
        np.testing.assert_allclose(got[:2], want[:2], rtol=1e-8)
    else:
        assert np.array_equal(single.bits(got), single.bits(want)), (got, want)


# ---------------------------------------------------------------- 4. the scoring rule on hand-built inputs
def _first_measurement(f, o, n):
    """Every slot visible, landmarks spread over a grid in front of the robot."""
    xy = np.array([[0.5 + 0.35 * (i % 5), -0.7 + 0.35 * (i // 5)] for i in range(n)]).reshape(-1)
    vis = np.ones(n, np.uint8)
    f.prediction((0.01, 0.02))
    o.prediction(0.01, 0.02)
    f.measurement(xy, vis)
    o.measurement(xy, vis)


def _between_gates(o, known_count, k):
    """A reading near landmark k whose smallest distance to the known landmarks lies in [1, 10) (dropped)."""
    lo, hi = 0.0, 1.0
    for _ in range(60):
        s = 0.5 * (lo + hi)
        z = robot_frame(o.state, k, (s, 0.0))
        d = min(o.maha(z[0], z[1], i) for i in range(known_count))
        if d < 4.0:
            lo = s
        else:
            hi = s
    z = robot_frame(o.state, k, (lo, 0.0))
    d = min(o.maha(z[0], z[1], i) for i in range(known_count))
    assert 1.0 + 1e-6 < d < 10.0 - 1e-6, d
    return z


@pytest.mark.parametrize("engine,n", FILTERS, ids=[f"{e}-{n}" for e, n in FILTERS])
def test_scoring_rule(gpu_pkg, engine, n):
    f, o = _make(gpu_pkg, engine, n), NoiseOracle(n)
    f.set_nis(True)
    assert f.last_nis().size == 0  # no call has run with NIS on yet
    _first_measurement(f, o, n)
    assert f.nis()["count"] == 0 and f.update_count == n
    assert np.array_equal(f.last_nis(), np.full(n, -1.0))  # the first measurement() scores nothing
    kc = 5
    known = np.zeros(n, np.uint8)
    known[:kc] = 1
    ko = known.copy()
    dropped = _between_gates(o, kc, 3)
    update = robot_frame(o.state, 2, (0.004, -0.003))
    far = np.array([-3.0, 2.5])  # behind the robot, far from every known landmark: creates landmark kc
    meas = np.stack([dropped, update, far])
    got = f.data_association(meas, known)
    a, cr = o.data_association(meas, ko)
    assert np.array_equal(got["assoc"], a) and np.array_equal(a, [-1, 2, kc]) and np.array_equal(cr, [0, 0, 1])
    assert np.array_equal(known, ko)
    v = f.last_nis()
    assert v[0] == -1.0 and v[2] == -1.0  # dropped between the gates; created by its own reading
    assert np.isfinite(v[1]) and abs(v[1] - o.values[-1]) <= NIS_RTOL * abs(o.values[-1]), (v[1], o.values)
    r = f.nis()
    assert r["count"] == 1 and r["stats"][0] == v[1]


# ---------------------------------------------------------------- 5. read-out semantics
@pytest.mark.parametrize("engine,n", FILTERS, ids=[f"{e}-{n}" for e, n in FILTERS])
def test_readout(gpu_pkg, engine, n):
    T = 6
    tk, tu = single.traces(gpu_pkg, n, T, seed=900 + n, m_max=M_MAX)
    f = _make(gpu_pkg, engine, n)
    out, cnt = np.zeros(4), np.zeros(1, np.int32)
    assert f._L.ekf_nis(f._h, out.ctypes.data, 0) == -3  # EKF_ERR_STATE: NIS never enabled
    assert f._L.ekf_last_nis(f._h, out.ctypes.data, cnt.ctypes.data) == -3
    with pytest.raises(gpu_pkg.EkfError):
        f.nis()
    assert f._L.ekf_nis(f._h, None, 0) != 0 and f._L.ekf_set_nis(None, 1) != 0
    f.set_nis(True)
    known = np.zeros(n, np.uint8)
    for t in range(3):
        single.step_known(f, tk, t)
        single.step_unknown(f, tu, t, known)
    s1 = f.nis()["stats"]
    assert s1[2] > 0 and np.array_equal(single.bits(f.nis()["stats"]), single.bits(s1))  # a read changes nothing
    # steps with NIS off leave the accumulators and the last call's values alone
    last = f.last_nis()
    f.set_nis(False)
    single.step_known(f, tk, 3)
    single.step_unknown(f, tu, 3, known)
    assert np.array_equal(single.bits(f.nis()["stats"]), single.bits(s1))
    assert np.array_equal(single.bits(f.last_nis()), single.bits(last))
    # a clone continues bit-identically, accumulators included
    f.set_nis(True)
    g, kg = f.clone(), known.copy()
    assert np.array_equal(single.bits(g.nis()["stats"]), single.bits(s1))
    for t in range(4, T):
        for h, k in ((f, known), (g, kg)):
            single.step_known(h, tk, t)
            single.step_unknown(h, tu, t, k)
    assert np.array_equal(single.bits(f.nis()["stats"]), single.bits(g.nis()["stats"]))
    assert np.array_equal(single.bits(f.last_nis()), single.bits(g.last_nis()))
    assert np.array_equal(single.bits(f.state), single.bits(g.state))
    assert np.array_equal(single.bits(f.sigma), single.bits(g.sigma))
    # reset zeroes after the read
    s2 = f.nis(reset=True)["stats"]
    assert s2[2] > s1[2]
    assert np.all(f.nis()["stats"] == 0)
    # clone of a filter that has NIS switched off carries the switch: its steps leave the accumulators alone
    f.set_nis(False)
    h = f.clone()
    single.step_known(h, tk, 0)
    assert np.all(h.nis()["stats"] == 0)


@pytest.mark.parametrize("n", [20, 33])
def test_toggle_with_prediction_deferred(gpu_pkg, n):
    """The fused engine defers prediction() into the next kernel; switching NIS on or off in between changes nothing
    else: same state, covariance, launches and accumulators as switching before the prediction."""
    T = 5
    tk, _ = single.traces(gpu_pkg, n, T, seed=950 + n, m_max=M_MAX)
    a, b = _make(gpu_pkg, "fused", n), _make(gpu_pkg, "fused", n)
    for t in range(T):  # by hand: set_nis() falls between prediction() and measurement()
        on = t % 2 == 0
        a.set_nis(on)
        a.prediction(tuple(tk["twists"][t, 0]))
        b.prediction(tuple(tk["twists"][t, 0]))
        b.set_nis(on)  # the prediction is still deferred here
        for f in (a, b):
            f.measurement(tk["xy"][t, 0], tk["vis"][t, 0])
    assert np.array_equal(single.bits(a.state), single.bits(b.state))
    assert np.array_equal(single.bits(a.sigma), single.bits(b.sigma))
    assert a.launch_count == b.launch_count
    assert np.array_equal(single.bits(a.nis()["stats"]), single.bits(b.nis()["stats"]))
    assert np.array_equal(single.bits(a.last_nis()), single.bits(b.last_nis()))
    assert a.nis()["count"] > 0
