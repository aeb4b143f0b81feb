"""Batches of filters with 65 to 1,024 landmarks (the "wide" batch engine, covariances in HBM).

Every filter of a wide batch must be bit-identical, in state and covariance, to a single streamed filter
(EKF_SLAM(n, engine=ENGINE_STREAM)) with set_carry_pending(False) driven with the same inputs, and within the usual
1e-9 of the CPU oracle."""
import ctypes

import numpy as np
import pytest

import _single as single
from _batch import grid_world, run_known, step_known
from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu

TOL = 1e-9
P = 14  # factor pairs per pass over a filter's covariance


def _trace(pkg, n, B, T, seed):
    tr = pkg.tracegen.simulate_known(grid_world(pkg, n), B, T, seed=seed)
    tr["twists"][T // 2, :, 0] = 1e-8  # the straight-line branch of the motion model
    return tr


@pytest.mark.parametrize("n", [65, 100, 256, 512, 1024])
def test_wide_batch_is_bit_identical_to_streamed_filters(gpu_pkg, n):
    B, T = 48, 20
    tr = _trace(gpu_pkg, n, B, T, seed=100 + n)
    bt = gpu_pkg.EKFBatch(B, n)
    assert bt.engine == gpu_pkg.ENGINE_STREAM
    run_known(gpu_pkg, bt, tr)
    states = bt.states()
    assert bt.update_count == int(tr["vis"].sum())
    rng = np.random.default_rng(n)
    for b in [0, B - 1] + list(rng.choice(np.arange(1, B - 1), 4, replace=False)):
        f = single.streamed(gpu_pkg, n, tr, b, range(T))
        assert np.array_equal(states[b], f.state), b
        assert np.array_equal(bt.sigma(b), f.sigma), b
    # oracle parity on a few filters
    for b in (0, B // 2):
        o = single.run_known(OracleEKF(n), tr, b)
        assert state_err(states[b], o.state) < TOL
        assert sigma_err(bt.sigma(b), o.sigma) < TOL


def test_wide_batch_more_corrections_than_one_group(gpu_pkg):
    """A first call with all 100 slots visible needs several passes over Sigma inside one step."""
    n, B, T = 100, 16, 6
    tr = _trace(gpu_pkg, n, B, T, seed=7)
    tr["vis"][0] = 1
    tr["vis"][3, : B // 2] = 1
    bt = gpu_pkg.EKFBatch(B, n)
    run_known(gpu_pkg, bt, tr)
    c = tr["vis"].sum(axis=2)
    assert bt.update_count == int(c.sum())
    assert bt.sweep_count == int(np.ceil(c / P).sum())
    states = bt.states()
    for b in (0, B // 2 - 1, B // 2, B - 1):
        f = single.streamed(gpu_pkg, n, tr, b, range(T))
        assert np.array_equal(states[b], f.state), b
        assert np.array_equal(bt.sigma(b), f.sigma), b


@pytest.mark.parametrize("n", [100, 256])
def test_wide_batch_marker_list_equals_dense_arrays(gpu_pkg, n):
    B, T = 40, 8
    tr = _trace(gpu_pkg, n, B, T, seed=31)
    dense, sparse = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    for t in range(T):
        tw = np.ascontiguousarray(tr["twists"][t])
        xy = np.ascontiguousarray(tr["xy"][t]) * tr["vis"][t].repeat(2, axis=1)  # unlisted slots read (0, 0)
        vis = np.ascontiguousarray(tr["vis"][t])
        dense.step_known(tw, xy, vis)
        sparse.step_known_sparse(tw, *gpu_pkg.marker_list(xy, vis))
    dense.sync(), sparse.sync()
    assert sparse.update_count == dense.update_count == int(tr["vis"].sum())
    assert sparse.sweep_count == dense.sweep_count
    assert np.array_equal(sparse.states(), dense.states())
    for b in (0, B // 2, B - 1):
        assert np.array_equal(sparse.sigma(b), dense.sigma(b))


def test_wide_batch_marker_list_needs_uint8_ids(gpu_pkg):
    B, n = 4, 257
    bt = gpu_pkg.EKFBatch(B, n)
    L = gpu_pkg._lib.load()
    tw = np.zeros((B, 2))
    off = np.zeros(B + 1, np.int32)
    rc = L.ekf_batch_step_known_sparse(bt._h, tw.ctypes.data, off.ctypes.data, None, None, 0)
    assert rc == -2  # EKF_ERR_UNSUPPORTED
    assert b"uint8" in L.ekf_last_error()
    assert bt.update_count == 0


def test_wide_batch_checkpoint_resume_is_bit_identical(gpu_pkg, tmp_path):
    n, B, T = 100, 24, 12
    tr = _trace(gpu_pkg, n, B, T, seed=5)
    a, b = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)
    for t in range(T // 2):
        step_known(gpu_pkg, a, tr, t)
    path = str(tmp_path / "wide.npz")
    a.save_checkpoint(path)
    b.load_checkpoint(path)
    assert b.update_count == a.update_count
    for t in range(T // 2, T):
        step_known(gpu_pkg, a, tr, t)
        step_known(gpu_pkg, b, tr, t)
    a.sync(), b.sync()
    assert np.array_equal(a.states(), b.states()) and a.update_count == b.update_count
    for f in (0, B - 1):
        assert np.array_equal(a.sigma(f), b.sigma(f))
    with pytest.raises(ValueError):
        gpu_pkg.EKFBatch(B + 1, n).restore(a.checkpoint())
    with pytest.raises(ValueError):
        gpu_pkg.EKFBatch(B, n + 1).restore(a.checkpoint())


def test_wide_batch_engine_boundaries(gpu_pkg):
    assert gpu_pkg.EKFBatch(2, 64).engine == gpu_pkg.ENGINE_FUSED
    assert gpu_pkg.EKFBatch(2, 65).engine == gpu_pkg.ENGINE_STREAM
    big = gpu_pkg.EKFBatch(2, 1024)
    assert big.engine == gpu_pkg.ENGINE_STREAM
    with pytest.raises(gpu_pkg.EkfError) as e:
        gpu_pkg.EKFBatch(2, 1025)
    assert e.value.code == -2 and "EKF_ENGINE_STREAM" in str(e.value)
    # unknown association is refused and leaves the batch as it was
    n, B = 100, 8
    tr = _trace(gpu_pkg, n, B, 2, seed=9)
    bt = gpu_pkg.EKFBatch(B, n)
    step_known(gpu_pkg, bt, tr, 0)
    before = bt.states()
    with pytest.raises(gpu_pkg.EkfError) as e:
        bt.step_unknown(np.ones((B, 2)), np.ones((B, 4, 2)), np.full(B, 4, np.int32), 4)
    assert e.value.code == -2
    assert np.array_equal(bt.states(), before)
    # a 1,024-landmark step (every slot visible on the first call: 74 groups of factors) gives the bits of two streamed
    # filters
    tw = np.full((1, 2, 2), 0.01)
    rng = np.random.default_rng(4)
    r, phi = rng.uniform(0.5, 2.0, (2, 1024)), rng.uniform(-np.pi, np.pi, (2, 1024))
    xy = np.stack([r * np.cos(phi), r * np.sin(phi)], axis=2).reshape(1, 2, 2048)
    one = {"twists": tw, "xy": xy, "vis": np.ones((1, 2, 1024), np.uint8)}
    run_known(gpu_pkg, big, one)
    assert big.update_count == 2 * 1024 and big.sweep_count == 2 * int(np.ceil(1024 / P))
    states = big.states()
    for b in range(2):
        f = single.streamed(gpu_pkg, 1024, one, b, range(1))
        assert np.array_equal(single.bits(states[b]), single.bits(f.state)), b
        assert np.array_equal(single.bits(big.sigma(b)), single.bits(f.sigma)), b


def test_wide_batch_getters(gpu_pkg):
    n, B, T = 100, 12, 5
    tr = _trace(gpu_pkg, n, B, T, seed=13)
    bt = gpu_pkg.EKFBatch(B, n)
    for t in range(T):
        step_known(gpu_pkg, bt, tr, t)
    states = bt.states()
    assert np.array_equal(bt.poses(), states[:, :3])
    err = bt.pose_error(tr["truth"][-1])
    assert err[3] == B and np.all(np.isfinite(err))
    N, ld = 3 + 2 * n, (3 + 2 * n + 15) // 16 * 16
    sig_ptr, sig_stride, st_ptr, st_stride = bt.device_pointers()
    assert sig_stride == N * ld and st_stride >= N and sig_ptr and st_ptr
    # the documented layout: filter b's row r starts sigma + (b * N * ld + r * ld) doubles
    L = gpu_pkg._lib.load()
    ns, nst = ctypes.c_int64(), ctypes.c_int64()
    gpu_pkg._lib.check(L.ekf_batch_checkpoint_size(bt._h, ctypes.byref(ns), ctypes.byref(nst)))
    assert ns.value == B * N * ld and nst.value == B * st_stride
    ck = bt.checkpoint()
    dense = ck["sigma_packed"].reshape(B, N, ld)
    for b in (0, B - 1):
        assert np.array_equal(dense[b, :, :N], bt.sigma(b))
    known = np.zeros((B, n), np.uint8)
    known[:, :3] = 1
    bt.known = known
    assert np.array_equal(bt.known, known)
    assert bt.launch_count >= T
