"""Consistency read-out of a batch (EKFBatch.marginals, nees, nees_dev) in all three Sigma layouts: tile (n = 20),
staircase (n <= 64) and wide (64 < n <= 1,024).

The marginals must be the stored entries of sigma(b) bit for bit; NEES must match numpy on the dense matrices; the
batch partial must be the sum of the per-filter values and bit-identical from one call to the next; the read-out must
leave the batch untouched."""
import numpy as np
import pytest

from _batch import grid_world, run_known, run_unknown, sms, unknown_trace

pytestmark = pytest.mark.gpu

RTOL = 1e-10


def _known_batch(pkg, n, B, T, seed):
    w = grid_world(pkg, n)
    tr = pkg.tracegen.simulate_known(w, B, T, seed=seed)
    bt = pkg.EKFBatch(B, n)
    run_known(pkg, bt, tr)
    return bt, tr, w


def _unknown_batch(pkg, n, B, T, seed, m_max):
    tr = unknown_trace(pkg, n, B, T, seed, m_max)
    bt = pkg.EKFBatch(B, n)
    run_unknown(bt, tr, m_max)
    return bt, tr


def _filters(B, seed):
    rng = np.random.default_rng(seed)
    mid = list(rng.choice(np.arange(1, B - 1), min(3, B - 2), replace=False)) if B > 2 else []
    return sorted({0, B - 1, *[int(v) for v in mid]})


def _assert_marginals_stored(bt, filters):
    pose, lm = bt.marginals()
    assert np.array_equal(pose, np.swapaxes(pose, 1, 2)) and np.array_equal(lm, np.swapaxes(lm, 2, 3))
    r = 3 + 2 * np.arange(bt.n)
    for b in filters:
        S = bt.sigma(b)
        iu = np.triu_indices(3)
        assert np.array_equal(pose[b][iu], S[:3, :3][iu]), b
        assert np.array_equal(lm[b, :, 0, 0], S[r, r]), b
        assert np.array_equal(lm[b, :, 0, 1], S[r, r + 1]), b
        assert np.array_equal(lm[b, :, 1, 1], S[r + 1, r + 1]), b


@pytest.mark.parametrize("n", [1, 20, 33, 48, 64, 65, 100, 1024])
def test_marginals_are_the_stored_entries_known(gpu_pkg, n):
    B = 3 if n == 1024 else 24
    bt, _, _ = _known_batch(gpu_pkg, n, B, 6, seed=40 + n)
    _assert_marginals_stored(bt, _filters(B, n))


@pytest.mark.parametrize("n", [20, 33])
def test_marginals_are_the_stored_entries_unknown(gpu_pkg, n):
    B = 24
    bt, _ = _unknown_batch(gpu_pkg, n, B, 8, seed=n, m_max=12)
    _assert_marginals_stored(bt, _filters(B, n))


def _sym_upper(M):
    return np.triu(M) + np.triu(M, 1).T


def _nees_numpy(pkg, bt, truth, lm_truth, b, states):
    """Per-filter (pose NEES or NaN, landmark NEES sum, count, singular landmarks) from the dense covariance."""
    S, st = bt.sigma(b), states[b]
    known, init = bt.known[b], bt.checkpoint()["init_flag"][b]
    P = _sym_upper(S[:3, :3])
    e = np.array([pkg.tracegen.normalize_angle(st[0] - truth[b, 2]), st[1] - truth[b, 0], st[2] - truth[b, 1]])
    try:
        np.linalg.cholesky(P)
        pose = float(e @ np.linalg.solve(P, e))
    except np.linalg.LinAlgError:
        pose = np.nan
    vals, singular = [], 0
    if lm_truth is not None:
        lt = lm_truth if lm_truth.ndim == 2 else lm_truth[b]
        for i in range(bt.n):
            if not (init or known[i]) or not np.all(np.isfinite(lt[i])):
                continue
            r = 3 + 2 * i
            L = _sym_upper(S[r:r + 2, r:r + 2])
            if not (L[0, 0] > 0 and np.linalg.det(L) > 0):
                singular += 1
                continue
            d = st[r:r + 2] - lt[i]
            vals.append(float(d @ np.linalg.solve(L, d)))
    return pose, vals, singular


def _lm_truth_for(pkg, w, n, B, per_filter, seed):
    nt = min(w.n_tubes, n)
    shared = np.full((n, 2), np.nan)
    shared[:nt, 0], shared[:nt, 1] = w.tubes_x[:nt], w.tubes_y[:nt]
    if not per_filter:
        shared[n // 2] = np.nan  # one slot not scored
        return shared
    rng = np.random.default_rng(seed)
    lt = shared[None] + rng.normal(0, 0.01, (B, n, 2))
    lt[rng.random((B, n)) < 0.2] = np.nan  # NaN truth entries are not scored
    return lt


@pytest.mark.parametrize("per_filter_truth", [False, True])
@pytest.mark.parametrize("n", [20, 33, 65])
def test_nees_matches_numpy(gpu_pkg, n, per_filter_truth):
    B = 40
    bt, tr, w = _known_batch(gpu_pkg, n, B, 8, seed=7 * n)
    truth = np.ascontiguousarray(tr["truth"][-1])
    lt = _lm_truth_for(gpu_pkg, w, n, B, per_filter_truth, seed=n)
    res = bt.nees(truth, lt, per_filter=True)
    states = bt.states()
    for b in _filters(B, n + 1):
        pose, vals, singular = _nees_numpy(gpu_pkg, bt, truth, lt, b, states)
        assert singular == 0
        np.testing.assert_allclose(res["pose_nees"][b], pose, rtol=RTOL)
        assert res["landmark_nees_count"][b] == len(vals)
        np.testing.assert_allclose(res["landmark_nees_sum"][b], sum(vals), rtol=RTOL)
    # every filter has seen measurement(): every slot with finite truth is scored
    expect = np.broadcast_to(np.isfinite(lt).all(axis=-1).sum(axis=-1), (B,))
    assert np.array_equal(res["landmark_nees_count"], expect)
    assert res["pose_singular"] == 0 and res["landmark_singular"] == 0


def test_nees_singular_landmark_block(gpu_pkg):
    """A landmark block with a zero variance (written through checkpoint/restore of the dense wide layout) is NaN,
    excluded, and counted as singular."""
    n, B = 65, 6
    bt, tr, w = _known_batch(gpu_pkg, n, B, 5, seed=3)
    ck = bt.checkpoint()
    N, ld = 3 + 2 * n, (3 + 2 * n + 15) // 16 * 16
    r = 3 + 2 * 7
    ck["sigma_packed"][2 * N * ld + r * ld + r] = 0.0
    bt.restore(ck)
    truth = np.ascontiguousarray(tr["truth"][-1])
    lt = _lm_truth_for(gpu_pkg, w, n, B, False, seed=1)
    res = bt.nees(truth, lt, per_filter=True)
    assert res["landmark_singular"] == 1
    scored = int(np.isfinite(lt).all(axis=1).sum())
    assert res["landmark_nees_count"][2] == scored - 1 and res["landmark_nees_count"][1] == scored
    pose, vals, singular = _nees_numpy(gpu_pkg, bt, truth, lt, 2, bt.states())
    assert singular == 1
    np.testing.assert_allclose(res["landmark_nees_sum"][2], sum(vals), rtol=RTOL)


@pytest.mark.parametrize("n", [20, 33, 100])
def test_before_the_first_step(gpu_pkg, n):
    """Sigma_0's robot block is zero: the pose is singular for every filter, and no landmark is scored before the
    first measurement()."""
    B = 10
    bt = gpu_pkg.EKFBatch(B, n)
    lt = np.zeros((n, 2))
    res = bt.nees(np.zeros((B, 3)), lt, per_filter=True)
    assert np.all(np.isnan(res["pose_nees"]))
    assert res["pose_singular"] == B and res["pose_count"] == 0
    assert res["landmark_count"] == 0 and res["landmark_singular"] == 0
    assert np.all(res["landmark_nees_count"] == 0)
    # known_list alone makes a slot count
    kn = np.zeros((B, n), np.uint8)
    kn[3, 0] = 1
    bt.known = kn
    res = bt.nees(np.zeros((B, 3)), lt, per_filter=True)
    assert res["landmark_count"] == 1 and res["landmark_nees_count"][3] == 1


def test_unknown_association_scores_known_slots_only(gpu_pkg):
    n, B, m_max = 20, 32, 6
    bt, tr = _unknown_batch(gpu_pkg, n, B, 10, seed=11, m_max=m_max)
    known = bt.known
    assert 0 < known.sum() < known.size
    states = bt.states()
    lt = states[:, 3:].reshape(B, n, 2) + 0.01  # finite truth for every slot; only the known slots may count
    truth = np.ascontiguousarray(tr["truth"][-1])
    res = bt.nees(truth, np.ascontiguousarray(lt), per_filter=True)
    assert np.array_equal(res["landmark_nees_count"], known.sum(axis=1))
    for b in _filters(B, 5):
        pose, vals, _ = _nees_numpy(gpu_pkg, bt, truth, lt, b, states)
        np.testing.assert_allclose(res["pose_nees"][b], pose, rtol=RTOL)
        np.testing.assert_allclose(res["landmark_nees_sum"][b], sum(vals), rtol=RTOL)


@pytest.mark.parametrize("n", [20, 33])
def test_batch_partials_are_the_per_filter_sums_and_repeat_bit_for_bit(gpu_pkg, n):
    """B above 64 warps per SM (more filters than any grid of the kernel has warps) and not a multiple of 8 warps."""
    B = 64 * sms() + 37
    T = 4
    w = grid_world(gpu_pkg, n)
    tr = gpu_pkg.tracegen.simulate_known(w, 61, T, seed=5)  # filter b runs trajectory b mod 61

    def rep(a):
        return np.ascontiguousarray(np.tile(a, (-(-B // 61),) + (1,) * (a.ndim - 1))[:B])

    bt = gpu_pkg.EKFBatch(B, n)
    for t in range(T):
        bt.step_known(rep(tr["twists"][t]), rep(tr["xy"][t]), rep(tr["vis"][t]))
    truth = rep(tr["truth"][-1]) + np.random.default_rng(0).normal(0, 0.01, (B, 3))
    lt = _lm_truth_for(gpu_pkg, w, n, B, True, seed=2)
    r1 = bt.nees(truth, lt, per_filter=True)
    r2 = bt.nees(truth, lt, per_filter=True)
    r3 = bt.nees(truth, lt)
    assert np.array_equal(r1["stats"], r2["stats"]) and np.array_equal(r1["stats"], r3["stats"])
    assert np.array_equal(r1["pose_nees"], r2["pose_nees"], equal_nan=True)
    s = r1["stats"]
    p = r1["pose_nees"][np.isfinite(r1["pose_nees"])]
    assert s[2] == p.size == B and s[6] == 0
    np.testing.assert_allclose(s[0], p.sum(), rtol=1e-12)
    np.testing.assert_allclose(s[1], (p * p).sum(), rtol=1e-12)
    np.testing.assert_allclose(s[3], r1["landmark_nees_sum"].sum(), rtol=1e-12)
    assert s[5] == r1["landmark_nees_count"].sum() == np.isfinite(lt).all(axis=-1).sum()


def test_device_path_matches_host_and_needs_no_sync(gpu_pkg):
    import torch
    n, B, K = 20, 256, 6
    w = gpu_pkg.tracegen.dense_world(n)

    def run(sync_each):
        sim = gpu_pkg.TubeWorld(w, B, seed=21)
        bt = gpu_pkg.EKFBatch(B, n)
        sim.use_stream(bt.stream)
        p = sim.device_pointers()
        lt = np.full((n, 2), np.nan)
        lt[:, 0], lt[:, 1] = w.tubes_x[:n], w.tubes_y[:n]
        d_lt = torch.from_numpy(lt).cuda()
        out = torch.zeros((K, 8), dtype=torch.float64, device="cuda")
        pf = torch.zeros((K, B, 3), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        host = []
        for k in range(K):
            sim.step_known()
            bt.step_known_dev(p["twists"], p["xy"], p["vis"])
            bt.nees_dev(p["truth"], out[k].data_ptr(), d_lt.data_ptr(), 0, pf[k].data_ptr())
            if sync_each:
                bt.sync()
                truth = sim.download()["truth"]
                host.append(bt.nees(truth, lt, per_filter=True))
        bt.sync()
        res = out.cpu().numpy(), pf.cpu().numpy(), host
        sim.close()
        bt.close()
        return res

    o_sync, pf_sync, host = run(True)
    o_async, pf_async, _ = run(False)
    assert np.array_equal(o_sync, o_async)
    assert np.array_equal(pf_sync, pf_async, equal_nan=True)
    for k in range(K):
        assert np.array_equal(o_sync[k], host[k]["stats"]), k
        assert np.array_equal(pf_sync[k][:, 0], host[k]["pose_nees"], equal_nan=True)
        assert np.array_equal(pf_sync[k][:, 1], host[k]["landmark_nees_sum"])
    assert o_sync[-1][2] == B and o_sync[-1][5] > 0


@pytest.mark.parametrize("n", [20, 33, 100])
def test_read_out_changes_nothing(gpu_pkg, n):
    B = 16
    bt, tr, w = _known_batch(gpu_pkg, n, B, 5, seed=9)
    before = bt.checkpoint()
    u0, s0 = bt.update_count, bt.sweep_count
    truth = np.ascontiguousarray(tr["truth"][-1])
    lt = _lm_truth_for(gpu_pkg, w, n, B, True, seed=4)
    for _ in range(2):
        bt.marginals()
        bt.nees(truth, lt, per_filter=True)
        bt.nees(truth)
    after = bt.checkpoint()
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    assert bt.update_count == u0 and bt.sweep_count == s0


def test_invalid_arguments_enqueue_nothing(gpu_pkg):
    n, B = 20, 8
    bt = gpu_pkg.EKFBatch(B, n)
    L = gpu_pkg._lib.load()
    truth = np.zeros((B, 3))
    lt = np.zeros((B, n, 2))
    out = np.zeros(8)
    c0 = bt.launch_count
    for fn in (L.ekf_batch_nees, L.ekf_batch_nees_dev):
        assert fn(bt._h, truth.ctypes.data, lt.ctypes.data, 2 * n + 1, None, out.ctypes.data) == -1
        assert fn(bt._h, truth.ctypes.data, lt.ctypes.data, n, None, out.ctypes.data) == -1
        assert fn(bt._h, None, lt.ctypes.data, 0, None, out.ctypes.data) == -1
        assert fn(bt._h, truth.ctypes.data, lt.ctypes.data, 0, None, None) == -1
        assert fn(None, truth.ctypes.data, lt.ctypes.data, 0, None, out.ctypes.data) == -1
    assert L.ekf_batch_get_marginals(None, out.ctypes.data, None) == -1
    assert bt.launch_count == c0
    with pytest.raises(ValueError):
        bt.nees(truth, np.zeros((n + 1, 2)))
    bt.nees(truth, lt)  # valid: one launch
    assert bt.launch_count == c0 + 1
