"""The persistent batch kernels beyond one resident wave, where a CTA carries several filters one after the other:
ekf_fused_tile_kernel<ASSOC> (n = 20; min(B, SMs x occupancy) single-warp CTAs) and k_wide_step (64 < n <= 1,024;
min(B, SMs) CTAs).  Code that only runs from a CTA's second filter on - staging the next filter's Sigma and inputs,
the mbarrier phase, the zero tails of the gathered rows, the association mirrors, the visible set, the wide engine's
dirty factor slots and sweep ring - is checked here, and so is the double-buffered input copy of back-to-back
host-fed steps.

The replica method: K trajectories are simulated and filter b runs trajectory b mod K.  Replicas of one trajectory
must be bit-identical in every word the engine keeps (checkpoint()), and only the K references go through the oracle
(or through a streamed filter, for the wide engine).  K is a prime larger than 32 that does not divide the SM count,
so no grid SMs x c (c <= 32) is a multiple of K and a filter's predecessor on its CTA always ran another
trajectory."""
import ctypes

import numpy as np
import pytest

import _single as single
from _batch import assert_clear, assert_replicas, assert_same_checkpoint, dev, grid_world, replicate, sms
from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu

TOL = 1e-9
K = 61
P = 14  # factor pairs per pass over a wide filter's covariance
NT = 20  # the tile kernel's map size
M_MAX = 40  # more readings than lanes
KNOWN_CLASSES = (0, 1, 2, 3, 7, 20)  # corrections per step of trajectory k's class k % 6 (7: each slot at p = 0.35)
WIDE_CLASSES = (0, 1, 13, 14, 15, 29)


def _assert_checkpoint_replicas(bt):
    ck = bt.checkpoint()
    for key in ("sigma_packed", "state", "init_flag", "known"):
        assert_replicas(ck[key], bt.B, K, key)
    assert_replicas(bt.states(), bt.B, K, "states()")
    for k in range(K):
        last = k + K * ((bt.B - 1 - k) // K)
        assert np.array_equal(single.bits(bt.sigma(last)), single.bits(bt.sigma(k))), (k, last)
    return ck


def _assert_tile_schedule(busy, sms):
    """busy [T, B]: whether filter b has corrections (or readings) at step t.  For every plausible tile grid SMs x c,
    some CTA runs a busy filter right after an idle one, and an idle one right after a busy one."""
    B = busy.shape[1]
    for c in range(1, 33):
        grid = sms * c
        assert grid % K != 0 and B >= 2 * grid, c  # two filters or more on every CTA, and never a replica
        prev, nxt = busy[:, :-grid], busy[:, grid:]
        assert (~prev & nxt).any() and (prev & ~nxt).any(), c


# ---------------------------------------------------------------- tile kernel, known association
T_KNOWN = 12


@pytest.fixture(scope="module")
def known_inputs(gpu_pkg):
    """K trajectories in a 5 x 4 grid world with every tube in sight, thinned per class.  A class with corrections
    lists every slot in the first call, which initialises each landmark at its reading; unlisted slots read (0, 0), as
    the marker list implies.  One step drives straight (the motion model's second branch)."""
    tg = gpu_pkg.tracegen
    w = tg.grid_world(5, 4, pitch=0.3, n_slots=NT, max_visible=3.0)
    tr = tg.simulate_known(w, K, T_KNOWN, seed=61)
    rng = np.random.default_rng(61)
    vis = np.zeros((T_KNOWN, K, NT), np.uint8)
    for k in range(K):
        c = KNOWN_CLASSES[k % 6]
        if c == 0:
            continue
        vis[0, k] = 1
        for t in range(1, T_KNOWN):
            if c == 7:
                vis[t, k] = rng.random(NT) < 0.35
            else:
                vis[t, k, rng.choice(NT, c, replace=False)] = 1
    tw = tr["twists"].copy()
    tw[T_KNOWN // 3, :, 0] = 1e-8
    return {"twists": tw, "xy": tr["xy"] * vis.repeat(2, axis=2), "vis": vis}


def _sparse_dev(bt, tw, off, ids, pts):
    """ekf_batch_step_known_sparse_dev (no Python wrapper): the marker list in device memory."""
    import torch
    d_tw, d_off, d_ids, d_pts = dev(tw), dev(off), dev(ids if ids.size else np.zeros(1, np.uint8)), dev(pts)
    torch.cuda.synchronize()
    rc = bt._L.ekf_batch_step_known_sparse_dev(bt._h, d_tw.data_ptr(), d_off.data_ptr(), d_ids.data_ptr(),
                                               d_pts.data_ptr(), ctypes.c_int64(int(off[-1])))
    bt.sync()  # the tensors may go once the step has read them
    assert rc == 0, bt._L.ekf_last_error()


def test_tile_known_replicas_in_every_input_form(gpu_pkg, known_inputs):
    """Dense host arrays, dense device pointers, and the marker list from host and device memory, each at
    B = 64 x SMs + 37: bit-identical replicas, the four forms bit-identical to each other, the K references against
    the oracle."""
    import torch
    B = 64 * sms() + 37
    tw, xy, vis = (replicate(known_inputs[k], B, K) for k in ("twists", "xy", "vis"))
    _assert_tile_schedule(vis.any(axis=2), sms())
    host, device, sp_host, sp_dev = (gpu_pkg.EKFBatch(B, NT) for _ in range(4))
    for t in range(T_KNOWN):
        host.step_known(tw[t], xy[t], vis[t])
        d_tw, d_xy, d_vis = dev(tw[t]), dev(xy[t]), dev(vis[t])
        torch.cuda.synchronize()
        device.step_known_dev(d_tw.data_ptr(), d_xy.data_ptr(), d_vis.data_ptr())
        device.sync()
        off, ids, pts = gpu_pkg.marker_list(xy[t], vis[t])
        assert (np.diff(off) == 0).any()  # some filters list no marker at all
        sp_host.step_known_sparse(tw[t], off, ids, pts)
        _sparse_dev(sp_dev, tw[t], off, ids, pts)
    host.sync(), sp_host.sync()
    assert host.update_count == int(vis.sum())
    ck = _assert_checkpoint_replicas(host)
    for other in (device, sp_host, sp_dev):
        assert_same_checkpoint(other.checkpoint(), ck)
    states = host.states()
    for k in range(K):
        o = single.run_known(OracleEKF(NT), known_inputs, k)
        assert state_err(states[k], o.state) < TOL, k
        assert sigma_err(host.sigma(k), o.sigma) < TOL, k


# ---------------------------------------------------------------- tile kernel, unknown association
T_UNKNOWN = 12


@pytest.fixture(scope="module")
def unknown_inputs(gpu_pkg):
    """49 tubes on a 7 x 7 grid, all within sight, for 20 slots: 40 readings a step, and the map fills.  Count classes:
    0; negative; above m_max; exactly m_max; mixed in [-2, m_max + 5]; one to three readings (the map fills slowly)."""
    tg = gpu_pkg.tracegen
    w = tg.grid_world(7, 7, pitch=0.45, max_visible=3.0)
    w.n_slots = NT
    tu = tg.simulate_unknown(w, K, T_UNKNOWN, seed=62, m_max=M_MAX)
    assert np.all(tu["count"] == M_MAX)
    rng = np.random.default_rng(62)
    count = np.zeros((T_UNKNOWN, K), np.int32)
    for k in range(K):
        cls = k % 6
        for t in range(T_UNKNOWN):
            count[t, k] = (0, -1 - t % 3, M_MAX + 1 + t, M_MAX, int(rng.integers(-2, M_MAX + 6)),
                           int(rng.integers(1, 4)))[cls]
    return {"twists": tu["twists"], "meas": tu["meas"], "count": count}


def test_tile_unknown_replicas_host_and_device(gpu_pkg, unknown_inputs):
    """ekf_fused_tile_kernel<true> at m_max = 40 and B = 64 x SMs + 37, through step_unknown(want_assoc=True) and
    step_unknown_dev with a device count array: bit-identical replicas in association outputs, known lists, state and
    Sigma; the K references against the oracle."""
    import torch
    B = 64 * sms() + 37
    tw, meas, cnt = (replicate(unknown_inputs[k], B, K) for k in ("twists", "meas", "count"))
    _assert_tile_schedule(cnt > 0, sms())
    host, device = gpu_pkg.EKFBatch(B, NT), gpu_pkg.EKFBatch(B, NT)
    assoc = []
    out = torch.empty((B, M_MAX), dtype=torch.int32, device="cuda")
    for t in range(T_UNKNOWN):
        assoc.append(host.step_unknown(tw[t], meas[t], cnt[t], M_MAX, want_assoc=True))
        d_tw, d_me, d_ct = dev(tw[t]), dev(meas[t]), dev(cnt[t])
        out.fill_(77)
        torch.cuda.synchronize()
        device.step_unknown_dev(d_tw.data_ptr(), d_me.data_ptr(), d_ct.data_ptr(), M_MAX, out.data_ptr())
        device.sync()
        assert np.array_equal(out.cpu().numpy(), assoc[t]), t
        assert_replicas(assoc[t], B, K, f"association outputs of step {t}")
    ck = _assert_checkpoint_replicas(host)
    assert_same_checkpoint(device.checkpoint(), ck)
    states, known = host.states(), host.known
    full = 0
    for k in range(K):
        o = OracleEKF(NT)
        kn = np.zeros(NT, np.uint8)
        for t, (a, dmin, sec, cr) in enumerate(single.run_unknown(o, unknown_inputs, kn, k)):
            m = len(a)
            assert_clear(dmin, sec)
            assert np.array_equal(assoc[t][k, :m], a), (k, t)
            assert np.all(assoc[t][k, m:] == -1), (k, t)
            full += int(np.sum((dmin >= 10.0) & (cr == 0)))
        assert np.array_equal(known[k], kn), k
        assert state_err(states[k], o.state) < TOL, k
        assert sigma_err(host.sigma(k), o.sigma) < TOL, k
    assert full > 0  # readings dropped because the map was full


# ---------------------------------------------------------------- wide engine
T_WIDE = 6


def _wide_inputs(pkg, n):
    """K trajectories on an n-landmark grid; a class with corrections lists every slot in the first call (all n
    corrections in one step), then WIDE_CLASSES[k % 6] random slots per step."""
    tr = pkg.tracegen.simulate_known(grid_world(pkg, n), K, T_WIDE, seed=n)
    rng = np.random.default_rng(n)
    vis = np.zeros((T_WIDE, K, n), np.uint8)
    for k in range(K):
        c = WIDE_CLASSES[k % 6]
        if c == 0:
            continue
        vis[0, k] = 1
        for t in range(1, T_WIDE):
            vis[t, k, rng.choice(n, c, replace=False)] = 1
    tw = tr["twists"].copy()
    tw[T_WIDE // 2, :, 0] = 1e-8
    return {"twists": tw, "xy": tr["xy"] * vis.repeat(2, axis=2), "vis": vis}


def _assert_wide_schedule(counts, sms):
    """counts [T, B] corrections per filter and step; the grid is min(B, SMs) (ekf_batch_create).  Some CTA runs a
    filter whose short group (c mod 14 > 0) is shorter than its predecessor's, and one where it is longer."""
    short = counts % P
    prev, nxt = short[:, :-sms], short[:, sms:]
    both = (prev > 0) & (nxt > 0)
    assert (both & (nxt < prev)).any() and (both & (nxt > prev)).any()


@pytest.mark.parametrize("n", [65, 256, 1024])
def test_wide_replicas_dense_and_marker_list(gpu_pkg, n):
    """At n = 1,024 (10 GB of Sigma, the size bench_wide_batch.py reports) there is no marker list (its ids are
    uint8), and a seeded third of the references, every class among them, is replayed through streamed filters."""
    B = 2 * sms() + 5
    ref = _wide_inputs(gpu_pkg, n)
    tw, xy, vis = (replicate(ref[k], B, K) for k in ("twists", "xy", "vis"))
    counts = vis.sum(axis=2)
    _assert_wide_schedule(counts, sms())
    dense = gpu_pkg.EKFBatch(B, n)
    sparse = gpu_pkg.EKFBatch(B, n) if n <= 256 else None
    assert dense.engine == gpu_pkg.ENGINE_STREAM
    for t in range(T_WIDE):
        dense.step_known(tw[t], xy[t], vis[t])
        if sparse is not None:
            sparse.step_known_sparse(tw[t], *gpu_pkg.marker_list(xy[t], vis[t]))
    dense.sync()
    assert dense.update_count == int(counts.sum())
    assert dense.sweep_count == int(np.ceil(counts / P).sum())
    ck = _assert_checkpoint_replicas(dense)
    if sparse is not None:
        sparse.sync()
        assert_same_checkpoint(sparse.checkpoint(), ck)
        assert sparse.sweep_count == dense.sweep_count
    del ck  # 10 GB of host memory at n = 1,024
    states = dense.states()
    refs = range(K) if n <= 256 else sorted(set(range(6)) | set(np.random.default_rng(n).choice(K, 15, replace=False)))
    for k in refs:
        f = single.streamed(gpu_pkg, n, ref, k, range(T_WIDE))
        assert np.array_equal(single.bits(states[k]), single.bits(f.state)), k
        assert np.array_equal(single.bits(dense.sigma(k)), single.bits(f.sigma)), k
        f.close()
    k = WIDE_CLASSES.index(29)
    o = single.run_known(OracleEKF(n), ref, k)
    assert state_err(states[k], o.state) < TOL
    assert sigma_err(dense.sigma(k), o.sigma) < TOL


# ---------------------------------------------------------------- back-to-back host-fed steps
# Step t + 2 reuses step t's input slot: its copy may start only once step t's kernel is done (ev_consumed), and the
# kernel of a step only once its own copy has landed (ev_copied).  To exercise that ordering, every buffer (pinned
# inputs, pose buffers, the batch itself: cudaMallocHost and cudaMalloc may synchronise) exists before the first step,
# and nothing between the steps waits for the device.
def _pinned(pkg, a):
    buf = pkg.PinnedBuffer(a.shape, a.dtype)
    buf.array[...] = a
    return buf


def _device_fed_reference(pkg, B, step_dev, device_inputs):
    """A batch fed from device memory and synchronised after every step: its checkpoint and its poses after each
    step."""
    import torch
    torch.cuda.synchronize()  # the inputs' copies (on torch's stream) have landed
    ref = pkg.EKFBatch(B, NT)
    poses = []
    for d in device_inputs:
        step_dev(ref, *(x.data_ptr() for x in d))
        ref.sync()
        poses.append(ref.poses())
    return ref.checkpoint(), poses


def _assert_back_to_back(bt, steps, pose_bufs, want_ck, want_poses):
    for step, buf in zip(steps, pose_bufs):  # nothing here waits for the device
        step()
        bt.poses_async(buf)
    bt.sync()
    assert_same_checkpoint(bt.checkpoint(), want_ck)
    for t, (got, want) in enumerate(zip(pose_bufs, want_poses)):
        assert np.array_equal(single.bits(got.array), single.bits(want)), t


def test_tile_known_back_to_back_host_steps(gpu_pkg, known_inputs):
    """Host-fed steps with one synchronisation at the end: every input in its own pinned buffer so that the copies are
    truly asynchronous, dense and marker-list steps alternating through the same two input slots, and the poses read
    back asynchronously after every step.  Reference: a batch fed from device memory, synchronised after each step."""
    B = 64 * sms() + 37
    tw, xy, vis = (replicate(known_inputs[k], B, K) for k in ("twists", "xy", "vis"))
    want_ck, want_poses = _device_fed_reference(
        gpu_pkg, B, lambda bt, *d: bt.step_known_dev(*d),
        [(dev(tw[t]), dev(xy[t]), dev(vis[t])) for t in range(T_KNOWN)])
    inputs = [[_pinned(gpu_pkg, a) for a in ((tw[t], xy[t], vis[t]) if t % 2 == 0 else
                                             (tw[t], *gpu_pkg.marker_list(xy[t], vis[t])))] for t in range(T_KNOWN)]
    pose_bufs = [gpu_pkg.PinnedBuffer((B, 3), np.float64) for _ in range(T_KNOWN)]
    bt = gpu_pkg.EKFBatch(B, NT)
    steps = [(lambda a=a: bt.step_known(*a)) if t % 2 == 0 else (lambda a=a: bt.step_known_sparse(*a))
             for t, a in enumerate(inputs)]
    _assert_back_to_back(bt, steps, pose_bufs, want_ck, want_poses)


def test_tile_unknown_back_to_back_host_steps(gpu_pkg, unknown_inputs):
    """As above for step_unknown without association outputs (which would synchronise).  The first step enlarges the
    reading slots to m_max and synchronises while nothing else is in flight."""
    B = 64 * sms() + 37
    tw, meas, cnt = (replicate(unknown_inputs[k], B, K) for k in ("twists", "meas", "count"))
    want_ck, want_poses = _device_fed_reference(
        gpu_pkg, B, lambda bt, *d: bt.step_unknown_dev(*d, M_MAX),
        [(dev(tw[t]), dev(meas[t]), dev(cnt[t])) for t in range(T_UNKNOWN)])
    inputs = [[_pinned(gpu_pkg, a) for a in (tw[t], meas[t], cnt[t])] for t in range(T_UNKNOWN)]
    pose_bufs = [gpu_pkg.PinnedBuffer((B, 3), np.float64) for _ in range(T_UNKNOWN)]
    bt = gpu_pkg.EKFBatch(B, NT)
    steps = [(lambda a=a: bt.step_unknown(*a, M_MAX)) for a in inputs]
    _assert_back_to_back(bt, steps, pose_bufs, want_ck, want_poses)
