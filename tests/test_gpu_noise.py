"""Per-filter process and measurement noise (Q, R): EKFBatch.set_noise / noise in the tile (n = 20), staircase
(n <= 64) and wide (64 < n <= 1,024) layouts, and EKF_SLAM.set_noise on the fused and streamed single filters.

The NOISE variants of the step kernels must give the default kernels' results when the reference values are set
explicitly, and follow tests/_noise_ref.py (the CPU oracle's arithmetic with Q and R as arguments) otherwise."""
import numpy as np
import pytest

import _single as single
from _batch import assert_same_checkpoint, known_trace, run_known, run_unknown, sms, step_known, unknown_trace
from _noise_ref import DEFAULT_NOISE, NoiseOracle
from _oracle import sigma_err, state_err

pytestmark = pytest.mark.gpu

M_MAX = 40
TOL = 1e-9
NIS_RTOL = 1e-8
# Noise classes of the parity tests.  A smaller R makes each correction remove more of Sigma, and the relative rounding
# error of what is left grows with it; these rows keep r >= 0.002, where the 1e-9 tolerance of the default holds.
GRID = np.array([[1e-4, 1e-4, 1e-4, 0.01, 0.01], [4e-4, 2e-4, 3e-4, 0.003, 0.002], [2e-5, 1e-3, 5e-4, 0.03, 0.004],
                 [0.0, 0.0, 0.0, 0.004, 0.002], [1e-3, 1e-5, 2e-4, 0.008, 0.05]])


def _rows(B):
    return GRID[np.arange(B) % len(GRID)]


def _check_filters(bt, refs, what):
    worst_s = worst_p = 0.0
    states = bt.states()
    for b, o in enumerate(refs):
        worst_s = max(worst_s, state_err(states[b], o.state))
        worst_p = max(worst_p, sigma_err(bt.sigma(b), o.sigma))
    print(f"{what}: state {worst_s:.2e}, sigma {worst_p:.2e}")
    assert worst_s < TOL and worst_p < TOL, (what, worst_s, worst_p)


# ---------------------------------------------------------------- 1. reference values set explicitly
CASES = [("tile-dense", 20, "dense"), ("tile-markers", 20, "markers"), ("tile-device", 20, "device"),
         ("tile-unknown", 20, "unknown"), ("stair-known", 33, "dense"), ("stair-unknown", 33, "unknown"),
         ("stair-device", 33, "device"), ("wide-dense", 100, "dense"), ("wide-markers", 100, "markers"),
         ("wide-device", 100, "device")]


@pytest.mark.parametrize("name,n,form", CASES, ids=[c[0] for c in CASES])
def test_reference_values_bit_identical(gpu_pkg, name, n, form):
    B, T = (48, 8) if n <= 64 else (6, 5)
    if form == "unknown":
        tr = unknown_trace(gpu_pkg, n, B, T, seed=n + 9, m_max=M_MAX)
    else:
        tr = known_trace(gpu_pkg, n, B, T, seed=n + 9)
    plain, explicit = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    explicit.set_noise([1e-4] * 3, [0.01] * 2)
    assert np.array_equal(explicit.noise(), np.tile(DEFAULT_NOISE, (B, 1)))
    if form == "unknown":
        assert np.array_equal(run_unknown(plain, tr, M_MAX), run_unknown(explicit, tr, M_MAX))
    else:
        run_known(gpu_pkg, plain, tr, form)
        run_known(gpu_pkg, explicit, tr, form)
    assert_same_checkpoint(plain.checkpoint(), explicit.checkpoint())
    assert plain.launch_count == explicit.launch_count


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_single_reference_values_bit_identical(gpu_pkg, engine):
    n, T = 20, 6
    eng = single.engine(gpu_pkg, engine)
    tk, tu = single.traces(gpu_pkg, n, T, seed=31, m_max=M_MAX)
    a, b = gpu_pkg.EKF_SLAM(n, engine=eng), gpu_pkg.EKF_SLAM(n, engine=eng)
    b.set_noise([1e-4] * 3, [0.01] * 2)
    ka, kb = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for t in range(T):
        assoc = []
        for f, k in ((a, ka), (b, kb)):
            single.step_known(f, tk, t)
            assoc.append(single.step_unknown(f, tu, t, k)["assoc"])
        assert np.array_equal(*assoc)
    assert np.array_equal(single.bits(a.state), single.bits(b.state))
    assert np.array_equal(single.bits(a.sigma), single.bits(b.sigma))
    assert a.calculate_maha_dis((0.3, 0.4), 2) == b.calculate_maha_dis((0.3, 0.4), 2)
    assert a.launch_count == b.launch_count


# ---------------------------------------------------------------- 2. per-filter noise against the reference
@pytest.mark.parametrize("n", [20, 33, 100, 256])
def test_known_matches_reference(gpu_pkg, n):
    B, T = (10, 8) if n <= 64 else (5, 5)
    tr = known_trace(gpu_pkg, n, B, T, seed=300 + n)
    rows = _rows(B)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_noise(rows[:, :3], rows[:, 3:])
    assert np.array_equal(bt.noise(), rows)
    bt.set_nis(True)
    run_known(gpu_pkg, bt, tr)
    refs = [single.run_known(NoiseOracle(n, rows[b]), tr, b) for b in range(B)]
    _check_filters(bt, refs, f"known n={n}")
    _check_nis(bt, refs, f"known n={n}")


def _check_nis(bt, refs, what):
    r = bt.nis(per_filter=True)
    assert np.array_equal(r["nis_count"][:len(refs)], [o.acc[2] for o in refs]), what
    for col, k in (("nis_sum", 0), ("nis_sq_sum", 1)):
        want = np.array([o.acc[k] for o in refs])
        err = np.abs(r[col][:len(refs)] - want) / np.maximum(np.abs(want), 1e-300)
        print(f"{what}: {col} worst relative deviation {err.max():.2e}")
        assert err.max() < NIS_RTOL, (what, col)


@pytest.mark.parametrize("n", [20, 33])
def test_unknown_matches_reference(gpu_pkg, n):
    B, T = 10, 10
    tr = unknown_trace(gpu_pkg, n, B, T, seed=400 + n, m_max=M_MAX)
    rows = _rows(B)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_noise(rows[:, :3], rows[:, 3:])
    bt.set_nis(True)
    assoc = run_unknown(bt, tr, M_MAX)
    refs = [NoiseOracle(n, rows[b]) for b in range(B)]
    known = [np.zeros(n, np.uint8) for _ in range(B)]
    for b, o in enumerate(refs):
        for t, (a, _) in enumerate(single.run_unknown(o, tr, known[b], b)):
            assert np.array_equal(a, assoc[t, b, :len(a)]), (t, b)
    assert np.array_equal(bt.known, np.stack(known))
    _check_filters(bt, refs, f"unknown n={n}")
    _check_nis(bt, refs, f"unknown n={n}")


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_single_matches_reference(gpu_pkg, engine):
    n, T = 20, 6
    tk, tu = single.traces(gpu_pkg, n, T, seed=41, m_max=M_MAX)
    row = GRID[1]
    f = gpu_pkg.EKF_SLAM(n, engine=single.engine(gpu_pkg, engine))
    f.set_noise(row[:3], row[3:])
    assert np.array_equal(f.noise, row)
    o = NoiseOracle(n, row)
    kf, ko = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for t in range(T):
        single.step_known(f, tk, t)
        a = single.step_unknown(f, tu, t, kf)["assoc"]
        single.step_known(o, tk, t)
        assert np.array_equal(a, single.step_unknown(o, tu, t, ko)[0]), t
    assert state_err(f.state, o.state) < TOL and sigma_err(f.sigma, o.sigma) < TOL
    for i in (0, 5, 13):
        d, want = f.calculate_maha_dis((0.3, -0.2), i), o.maha(0.3, -0.2, i)
        assert abs(d - want) <= TOL * max(1.0, abs(want)), (i, d, want)


@pytest.mark.parametrize("n", [100, 256])
def test_wide_bit_identical_to_streamed(gpu_pkg, n):
    B, T = 3, 4
    tr = known_trace(gpu_pkg, n, B, T, seed=500 + n)
    rows = _rows(B)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_noise(rows[:, :3], rows[:, 3:])
    run_known(gpu_pkg, bt, tr)
    for b in range(B):
        f = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
        f.set_carry_pending(False)
        f.set_noise(rows[b, :3], rows[b, 3:])
        single.run_known(f, tr, b)
        assert np.array_equal(single.bits(f.state), single.bits(bt.states()[b])), b
        assert np.array_equal(single.bits(f.sigma), single.bits(bt.sigma(b))), b


# ---------------------------------------------------------------- 3. several filters per persistent CTA
@pytest.mark.parametrize("n,form", [(20, "known"), (20, "unknown"), (33, "known"), (65, "known")])
def test_noise_classes_over_replicas(gpu_pkg, n, form):
    """One trajectory for every filter, K noise classes permuted over a batch beyond one resident wave: every replica
    is bit-identical to its class's first filter, and the class representatives match the reference."""
    K = len(GRID)
    B = (2 * sms() + 5) if n > 64 else (64 * sms() + 37)
    T = 4 if n > 64 else 8
    cls = np.random.default_rng(n).permutation(np.arange(B) % K)
    if form == "unknown":
        one = unknown_trace(gpu_pkg, n, 1, T, seed=600 + n, m_max=M_MAX)
    else:
        one = known_trace(gpu_pkg, n, 1, T, seed=600 + n)
    tr = {k: np.ascontiguousarray(np.repeat(v, B, axis=1)) for k, v in one.items() if k in ("twists", "xy", "vis", "meas", "count")}
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_noise(GRID[cls, :3], GRID[cls, 3:])
    if form == "unknown":
        run_unknown(bt, tr, M_MAX)
    else:
        run_known(gpu_pkg, bt, tr)
    st = single.bits(bt.states())
    reps = [int(np.flatnonzero(cls == k)[0]) for k in range(K)]
    for k in range(K):
        members = np.flatnonzero(cls == k)
        assert (st[members] == st[reps[k]]).all(), k
    for k in range(K):
        o = NoiseOracle(n, GRID[k])
        if form == "unknown":
            single.run_unknown(o, one, np.zeros(n, np.uint8))
        else:
            single.run_known(o, one)
        assert state_err(bt.states()[reps[k]], o.state) < TOL and sigma_err(bt.sigma(reps[k]), o.sigma) < TOL, k
    assert len(set(tuple(st[r]) for r in reps)) == K  # the classes really differ


# ---------------------------------------------------------------- 4. changing the noise mid-run
@pytest.mark.parametrize("n", [20, 33, 100])
def test_noise_changed_mid_run(gpu_pkg, n):
    B, T = 4, 6
    tr = known_trace(gpu_pkg, n, B, T, seed=700 + n)
    bt = gpu_pkg.EKFBatch(B, n)
    refs = [NoiseOracle(n) for _ in range(B)]
    for t in range(T):
        if t == 3:
            bt.set_noise(_rows(B)[:, :3], _rows(B)[:, 3:])
            for b, o in enumerate(refs):
                o.set_noise(_rows(B)[b])
        if t == 5:
            bt.set_noise()
            for o in refs:
                o.set_noise(DEFAULT_NOISE)
        step_known(gpu_pkg, bt, tr, t, "dense")
        for b, o in enumerate(refs):
            single.step_known(o, tr, t, b)
    bt.sync()
    _check_filters(bt, refs, f"mid-run n={n}")


@pytest.mark.parametrize("engine", ["fused", "stream"])
def test_single_noise_changed_with_prediction_pending(gpu_pkg, engine):
    """prediction(), then set_noise(), then measurement(): the prediction uses the old Q (the fused engine still holds
    it back when set_noise() is called), the corrections the new R."""
    n, T = 20, 5
    tk = known_trace(gpu_pkg, n, 1, T, seed=801)
    f, o = gpu_pkg.EKF_SLAM(n, engine=single.engine(gpu_pkg, engine)), NoiseOracle(n)
    for t in range(T):  # by hand: set_noise() falls between prediction() and measurement()
        f.prediction(tuple(tk["twists"][t, 0]))
        o.prediction(*tk["twists"][t, 0])
        row = GRID[1 + t % 4]
        f.set_noise(row[:3], row[3:])
        o.set_noise(row)
        f.measurement(tk["xy"][t, 0], tk["vis"][t, 0])
        o.measurement(tk["xy"][t, 0], tk["vis"][t, 0])
    assert state_err(f.state, o.state) < TOL and sigma_err(f.sigma, o.sigma) < TOL


# ---------------------------------------------------------------- 5. configuration handling
def test_broadcast_clone_and_checkpoints(gpu_pkg):
    n, B, T = 20, 16, 5
    tr = known_trace(gpu_pkg, n, B, T, seed=901)
    row = GRID[2]
    shared, per = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    shared.set_noise(row[:3], row[3:])
    per.set_noise(np.tile(row[:3], (B, 1)), np.tile(row[3:], (B, 1)))
    run_known(gpu_pkg, shared, tr)
    run_known(gpu_pkg, per, tr)
    assert_same_checkpoint(shared.checkpoint(), per.checkpoint())
    # checkpoints carry no noise: a restored batch keeps its own setting, a fresh one the reference values
    ck = shared.checkpoint()
    fresh = gpu_pkg.EKFBatch(B, n)
    fresh.restore(ck)
    assert np.array_equal(fresh.noise(), np.tile(DEFAULT_NOISE, (B, 1)))
    per.set_noise(GRID[1, :3], GRID[1, 3:])
    per.restore(ck)
    assert np.array_equal(per.noise(), np.tile(GRID[1], (B, 1)))
    for eng in (gpu_pkg.ENGINE_FUSED, gpu_pkg.ENGINE_STREAM):
        f = gpu_pkg.EKF_SLAM(n, engine=eng)
        f.set_noise(row[:3], row[3:])
        f.prediction((0.01, 0.02))
        g = f.clone()
        assert np.array_equal(g.noise, row)
        for h in (f, g):
            h.prediction(tuple(tr["twists"][1, 0]))
            h.measurement(tr["xy"][0, 0], tr["vis"][0, 0])
        assert np.array_equal(single.bits(f.sigma), single.bits(g.sigma))
        f.set_noise()
        assert np.array_equal(f.noise, DEFAULT_NOISE)


@pytest.mark.parametrize("bad", [(np.nan, 1e-4, 1e-4, 0.01, 0.01), (1e-4, -1e-6, 1e-4, 0.01, 0.01),
                                 (1e-4, 1e-4, 1e-4, 0.0, 0.01), (1e-4, 1e-4, 1e-4, 0.01, np.inf)],
                         ids=["nan", "negative-q", "zero-r", "inf-r"])
def test_invalid_rows_rejected(gpu_pkg, bad):
    n, B = 20, 8
    bad = np.array(bad)
    bt = gpu_pkg.EKFBatch(B, n)
    rows = _rows(B)
    bt.set_noise(rows[:, :3], rows[:, 3:])
    before = bt.checkpoint()
    mixed = rows.copy()
    mixed[5] = bad
    for q, r in ((mixed[:, :3], mixed[:, 3:]), (bad[:3], bad[3:])):
        with pytest.raises(gpu_pkg.EkfError):
            bt.set_noise(q, r)
        assert np.array_equal(bt.noise(), rows)
    assert_same_checkpoint(before, bt.checkpoint())
    for eng in (gpu_pkg.ENGINE_FUSED, gpu_pkg.ENGINE_STREAM):
        f = gpu_pkg.EKF_SLAM(n, engine=eng)
        f.set_noise(GRID[1, :3], GRID[1, 3:])
        with pytest.raises(gpu_pkg.EkfError):
            f.set_noise(bad[:3], bad[3:])
        assert np.array_equal(f.noise, GRID[1])
