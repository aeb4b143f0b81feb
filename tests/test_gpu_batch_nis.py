"""NIS (normalised innovation squared) of batch filters: EKFBatch.set_nis / nis / nis_dev in the tile (n = 20),
staircase (n <= 64) and wide (64 < n <= 1,024) layouts.

NIS = nu^T S^-1 nu of every scored correction, accumulated per filter as {sum, sum of squares, #scored, #non-finite}
by the NIS variants of the step kernels.  The tests check that the variants leave the filters bit-identical, that the
accumulators match the numpy restatement of the CPU oracle (tests/_noise_ref.py, at the reference noise), the scoring
rule, bit-identical replicas when persistent CTAs carry several filters, and the read-out verbs."""
import numpy as np
import pytest

import _single as single
from _batch import (assert_replicas, assert_same_checkpoint, known_trace, replicate, run_known, run_unknown, sms,
                    step_known, unknown_trace)
from _noise_ref import NoiseOracle

pytestmark = pytest.mark.gpu

K = 61  # trajectories of the several-filters-per-CTA layout: filter b runs trajectory b mod K
M_MAX = 40
NIS_RTOL = 1e-8  # sums against the numpy reference; observed deviations are printed (state parity is 1e-11)


# ---------------------------------------------------------------- 1. the NIS variants do not change the filters
CASES = [("tile-dense", 20, "dense"), ("tile-markers", 20, "markers"), ("tile-device", 20, "device"),
         ("tile-unknown", 20, "unknown"), ("stair-known", 33, "dense"), ("stair-unknown", 33, "unknown"),
         ("wide-dense", 100, "dense"), ("wide-markers", 100, "markers")]


@pytest.mark.parametrize("name,n,form", CASES, ids=[c[0] for c in CASES])
def test_nis_leaves_filters_unchanged(gpu_pkg, name, n, form):
    B, T = (48, 8) if n <= 64 else (6, 5)
    if form == "unknown":
        tr = unknown_trace(gpu_pkg, n, B, T, seed=n + 5, m_max=M_MAX)
    else:
        tr = known_trace(gpu_pkg, n, B, T, seed=n + 5)
    plain, scored = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    scored.set_nis(True)
    if form == "unknown":
        a, b = run_unknown(plain, tr, M_MAX), run_unknown(scored, tr, M_MAX)
        assert np.array_equal(a, b)
    else:
        run_known(gpu_pkg, plain, tr, form)
        run_known(gpu_pkg, scored, tr, form)
    assert_same_checkpoint(plain.checkpoint(), scored.checkpoint())
    assert plain.update_count == scored.update_count
    assert plain.launch_count == scored.launch_count
    r = scored.nis(per_filter=True)
    assert r["count"] > 0 and r["nonfinite"] == 0


# ---------------------------------------------------------------- 2. parity with the numpy reference
def _compare(res, refs, what):
    cnt = np.array([o.acc[2] for o in refs])
    assert np.array_equal(res["nis_count"][:len(refs)], cnt), what
    assert np.all(res["nis_nonfinite"][:len(refs)] == 0), what
    worst = 0.0
    for k, col in ((0, "nis_sum"), (1, "nis_sq_sum")):
        want = np.array([o.acc[k] for o in refs])
        err = np.abs(res[col][:len(refs)] - want) / np.maximum(np.abs(want), 1e-300)
        err[want == 0] = np.abs(res[col][:len(refs)][want == 0])
        worst = max(worst, float(err.max()))
    print(f"{what}: NIS sums vs numpy reference, worst relative deviation {worst:.2e}, scored {int(cnt.sum())}")
    assert worst < NIS_RTOL, (what, worst)


@pytest.mark.parametrize("n", [20, 33, 64, 100, 256])
def test_nis_known_matches_reference(gpu_pkg, n):
    B, T = (8, 8) if n <= 64 else (3, 5)
    tr = known_trace(gpu_pkg, n, B, T, seed=100 + n)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_nis(True)
    run_known(gpu_pkg, bt, tr, "dense")
    refs = [single.run_known(NoiseOracle(n), tr, b) for b in range(B)]
    _compare(bt.nis(per_filter=True), refs, f"known n={n}")


@pytest.mark.parametrize("n", [20, 33])
def test_nis_unknown_matches_reference(gpu_pkg, n):
    B, T = 8, 10
    tr = unknown_trace(gpu_pkg, n, B, T, seed=200 + n, m_max=M_MAX)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_nis(True)
    assoc = run_unknown(bt, tr, M_MAX)
    refs = [NoiseOracle(n) for _ in range(B)]
    created = dropped = 0
    for b, o in enumerate(refs):
        for t, (a, c) in enumerate(single.run_unknown(o, tr, np.zeros(n, np.uint8), b)):
            assert np.array_equal(a, assoc[t, b, :len(a)]), (t, b)
            created += int(c.sum())
            dropped += int((a < 0).sum())
    assert created > 0 and dropped > 0  # the rule's exceptions are exercised: new landmarks and readings between gates
    _compare(bt.nis(per_filter=True), refs, f"unknown n={n}")


# ---------------------------------------------------------------- 3. scoring rule
@pytest.mark.parametrize("n", [20, 33, 100])
def test_first_step_and_set_nis_off_score_nothing(gpu_pkg, n):
    B, T = 6, 4
    tr = known_trace(gpu_pkg, n, B, T, seed=7, p_vis=1.0)
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_nis(True)
    step_known(gpu_pkg, bt, tr, 0)
    r = bt.nis(per_filter=True)
    assert bt.update_count > 0
    assert np.all(r["stats"] == 0) and np.all(r["nis_count"] == 0)
    step_known(gpu_pkg, bt, tr, 1)
    after = bt.nis(per_filter=True)
    assert np.all(after["nis_count"] == tr["vis"][1].sum(axis=1))
    bt.set_nis(False)  # the plain kernels again; the accumulators are kept
    step_known(gpu_pkg, bt, tr, 2)
    assert np.array_equal(bt.nis()["stats"], after["stats"])
    bt.set_nis(True)
    step_known(gpu_pkg, bt, tr, 3)
    assert bt.nis()["count"] == after["count"] + int(tr["vis"][3].sum())


@pytest.mark.parametrize("n", [20, 33])
def test_created_landmarks_score_nothing(gpu_pkg, n):
    """One reading per filter on a fresh map: it creates landmark 0 and corrects it, unscored."""
    B = 8
    rng = np.random.default_rng(n)
    meas = np.zeros((B, M_MAX, 2))
    meas[:, 0] = rng.uniform(0.5, 1.5, (B, 2))
    bt = gpu_pkg.EKFBatch(B, n)
    bt.set_nis(True)
    a = bt.step_unknown(np.full((B, 2), 0.01), meas, np.ones(B, np.int32), M_MAX, want_assoc=True)
    assert np.all(a[:, 0] == 0) and bt.update_count == B
    assert np.all(bt.nis()["stats"] == 0)


# ---------------------------------------------------------------- 4. several filters per persistent CTA
def _per_filter(bt):
    r = bt.nis(per_filter=True)
    return np.stack([r["nis_sum"], r["nis_sq_sum"], r["nis_count"], r["nis_nonfinite"]], axis=1)


def test_tile_replicas_known_and_unknown(gpu_pkg):
    B = 64 * sms() + 37
    tk = known_trace(gpu_pkg, 20, K, 10, seed=61)
    bt = gpu_pkg.EKFBatch(B, 20)
    bt.set_nis(True)
    run_known(gpu_pkg, bt, {k: replicate(v, B, K) for k, v in tk.items()}, "dense")
    pf = _per_filter(bt)
    assert pf[:, 2].sum() > 0
    assert_replicas(pf, B, K, "tile known")
    tu = unknown_trace(gpu_pkg, 20, K, 10, seed=62, m_max=M_MAX)
    bu = gpu_pkg.EKFBatch(B, 20)
    bu.set_nis(True)
    run_unknown(bu, {k: replicate(tu[k], B, K) for k in ("twists", "meas", "count")}, M_MAX)
    pf = _per_filter(bu)
    assert pf[:, 2].sum() > 0
    assert_replicas(pf, B, K, "tile unknown")


def test_wide_replicas(gpu_pkg):
    B = 2 * sms() + 5
    tk = known_trace(gpu_pkg, 65, K, 4, seed=65, p_vis=0.2)
    bt = gpu_pkg.EKFBatch(B, 65)
    bt.set_nis(True)
    run_known(gpu_pkg, bt, {k: replicate(v, B, K) for k, v in tk.items()}, "dense")
    pf = _per_filter(bt)
    assert pf[:, 2].sum() > 0
    assert_replicas(pf, B, K, "wide")


def test_back_to_back_host_steps(gpu_pkg):
    """Host-fed steps from pinned buffers with a single synchronisation at the end give the accumulators of a batch fed
    from device memory and synchronised after every step."""
    B, T = 64 * sms() + 37, 8
    tk = {k: replicate(v, B, K) for k, v in known_trace(gpu_pkg, 20, K, T, seed=63).items()}
    ref = gpu_pkg.EKFBatch(B, 20)
    ref.set_nis(True)
    run_known(gpu_pkg, ref, tk, "device")
    bufs = []
    for t in range(T):
        row = []
        for a in (tk["twists"][t], tk["xy"][t], tk["vis"][t]):
            p = gpu_pkg.PinnedBuffer(a.shape, a.dtype)
            p.array[...] = a
            row.append(p)
        bufs.append(row)
    bt = gpu_pkg.EKFBatch(B, 20)
    bt.set_nis(True)
    for row in bufs:
        bt.step_known(*row)
    bt.sync()
    assert np.array_equal(single.bits(_per_filter(bt)), single.bits(_per_filter(ref)))


# ---------------------------------------------------------------- 5. read-out
def test_readout(gpu_pkg):
    import torch
    B, T, n = 40, 6, 33
    tr = known_trace(gpu_pkg, n, B, T, seed=9)
    bt = gpu_pkg.EKFBatch(B, n)
    with pytest.raises(gpu_pkg.EkfError):
        bt.nis()  # never enabled
    bt.set_nis(True)
    run_known(gpu_pkg, bt, tr, "dense")
    r1, r2 = bt.nis(per_filter=True), bt.nis(per_filter=True)
    assert np.array_equal(single.bits(r1["stats"]), single.bits(r2["stats"]))
    assert np.array_equal(single.bits(r1["nis_sum"]), single.bits(r2["nis_sum"]))
    assert r1["stats"][2] == r1["nis_count"].sum() and r1["stats"][3] == 0
    np.testing.assert_allclose(r1["stats"][0], r1["nis_sum"].sum(), rtol=1e-12)
    np.testing.assert_allclose(r1["stats"][1], r1["nis_sq_sum"].sum(), rtol=1e-12)
    assert np.isfinite(r1["anis"]) and r1["bounds_95"][0] < 2.0 < r1["bounds_95"][1]
    # device read-out without a synchronisation, then reset
    d_out, d_pf = torch.zeros(4, dtype=torch.float64, device="cuda"), torch.zeros(B, 4, dtype=torch.float64, device="cuda")
    bt.nis_dev(d_out.data_ptr(), d_pf.data_ptr(), reset=True)
    bt.sync()
    assert np.array_equal(single.bits(d_out.cpu().numpy()), single.bits(r1["stats"]))
    assert np.array_equal(single.bits(d_pf.cpu().numpy()[:, 0]), single.bits(r1["nis_sum"]))
    assert np.all(bt.nis()["stats"] == 0)
    # a null out4 is refused
    assert bt._L.ekf_batch_nis(bt._h, None, None, 0) != 0
    assert bt._L.ekf_batch_nis_dev(bt._h, None, None, 0) != 0
    assert bt._L.ekf_batch_set_nis(None, 1) != 0


@pytest.mark.parametrize("n", [20, 33])
def test_nan_covariance_counts_nonfinite(gpu_pkg, n):
    B, T = 8, 5
    tr = known_trace(gpu_pkg, n, B, T, seed=11, p_vis=1.0)
    a, b = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    for bt in (a, b):
        step_known(gpu_pkg, bt, tr, 0)
        bt.sync()
    ck = b.checkpoint()
    sig = ck["sigma_packed"].reshape(B, -1)
    bad = 3
    sig[bad, 960 if n == 20 else 0] = np.nan  # Sigma[0][0] of filter 3 (tile: the robot rows follow 960 fragments)
    b.restore(ck)
    assert np.isnan(b.sigma(bad)[0, 0])
    for bt in (a, b):
        bt.set_nis(True)
        for t in range(1, T):
            step_known(gpu_pkg, bt, tr, t)
        bt.sync()
    pa, pb = _per_filter(a), _per_filter(b)
    others = np.arange(B) != bad
    assert np.array_equal(single.bits(pa[others]), single.bits(pb[others]))
    assert pb[bad, 3] == tr["vis"][1:, bad].sum() and pb[bad, 2] == 0 and pb[bad, 0] == 0
