"""The batch engine for maps of up to 64 landmarks other than n = 20: ekf_fused_sym_kernel, which keeps each filter's
covariance in the packed symmetric staircase layout of csrc/ekf_fused_sym.cuh, against the CPU oracle.

Its code depends on the size in ways the n = 20 tile kernel never sees: the staircase offsets where N = 3 + 2n crosses a
16-row block, landmarks whose two rows 3+2i and 4+2i fall into different 16-row blocks (i = 6, 14, 22, ...), the second
visibility word for ids 32..63, the fifth column slot per lane (N = 129..131), and more than one landmark per lane in
the association scan (n > 32).  The sizes below put every one of those on an input.  Also here: the batch's clamping
of the per-filter measurement count (both batch kernels)."""
import numpy as np
import pytest

import _single as single
from _batch import assert_clear, dev, robot_frame, run_known, run_unknown, stair_row_base, stair_strides, step_known
from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu

TOL = 1e-9


# ---------------------------------------------------------------- staircase layout (formulas of ekf_fused_sym.cuh)
def pack_staircase(dense, N):
    """Dense N x N -> the stored part of the staircase: row r keeps the columns [16 floor(r / 16), N)."""
    out = np.zeros(stair_row_base(N, N))
    for r in range(N):
        c0 = r & ~15
        base = stair_row_base(r, N)
        out[base:base + N - c0] = dense[r, c0:]
    return out


def _grid_world(pkg, n, pitch=0.3):
    nx = int(np.ceil(np.sqrt(n)))
    w = pkg.tracegen.grid_world(nx, -(-n // nx), pitch=pitch, n_slots=n, max_visible=3.0)
    w.tubes_x, w.tubes_y = w.tubes_x[:n], w.tubes_y[:n]
    return w


def _known_trace(pkg, n, B, T, seed):
    """Every landmark within sight, thinned at random per filter and step so that the visible sets differ; the first
    call only initialises (nothing visible) and one step drives straight (the motion model's second branch)."""
    tr = pkg.tracegen.simulate_known(_grid_world(pkg, n), B, T, seed=seed)
    rng = np.random.default_rng(seed)
    tr["vis"] = (tr["vis"] & (rng.random(tr["vis"].shape) < 0.6)).astype(np.uint8)
    tr["twists"][T // 3, :, 0] = 1e-8
    return tr


def _picks(B, seed):
    return [0, B - 1] + [int(v) for v in np.random.default_rng(seed).choice(np.arange(1, B - 1), 2, replace=False)]


# N = 5, 15, 17, 31, 33, 35, 45, 65, 67, 69, 97, 127, 129, 131: both sides of every 16-row and 32-column boundary
@pytest.mark.parametrize("n", [1, 6, 7, 14, 15, 16, 21, 31, 32, 33, 47, 62, 63, 64])
def test_known_association_dense_matches_oracle(gpu_pkg, n):
    B, T = 33, 16
    tr = _known_trace(gpu_pkg, n, B, T, seed=300 + n)
    assert tr["vis"][1:].any(axis=(0, 1)).all()  # every slot is corrected at least once
    bt = gpu_pkg.EKFBatch(B, n)
    assert bt.engine == gpu_pkg.ENGINE_FUSED
    run_known(gpu_pkg, bt, tr)
    assert bt.update_count == int(tr["vis"].sum())
    states = bt.states()
    for b in _picks(B, n):
        o = single.run_known(OracleEKF(n), tr, b)
        assert state_err(states[b], o.state) < TOL, b
        assert sigma_err(bt.sigma(b), o.sigma) < TOL, b


def _marker_list_with_strays(xy, vis, n, t):
    """The marker list of dense [B, 2n] / [B, n] arrays, where every third filter also lists a marker with an id >= n
    (which the batch ignores) in the middle of its list."""
    B = vis.shape[0]
    offsets = np.zeros(B + 1, np.int32)
    ids, pts = [], []
    for b in range(B):
        seen = list(np.flatnonzero(vis[b]))
        if b % 3 == 0:
            seen.insert(len(seen) // 2, n + (b + t) % 7)
        for i in seen:
            ids.append(i)
            pts.append(xy[b, 2 * i:2 * i + 2] if i < n else (0.4, -0.2))
        offsets[b + 1] = len(ids)
    return offsets, np.array(ids, np.uint8), np.ascontiguousarray(np.array(pts, np.float64).reshape(-1, 2))


@pytest.mark.parametrize("n", [7, 33, 64])
def test_marker_list_matches_oracle(gpu_pkg, n):
    """The marker list through the staircase kernel against the oracle fed the dense arrays the list stands for
    (unlisted slots read (0, 0)): the first call lists a random subset and initialises every slot, one step lists
    only ids >= 32 (none for n = 7), and stray ids >= n are ignored.  A slot left out of the first call starts at the
    robot's position and is never listed again: its first correction would be taken a few millimetres from the robot,
    where H_j is so large that rounding no longer stays within the tolerance."""
    B, T = 16, 10
    tr = _known_trace(gpu_pkg, n, B, T, seed=400 + n)
    rng = np.random.default_rng(n)
    vis = tr["vis"].copy()
    vis[0] = rng.random((B, n)) < 0.75
    vis[1:] &= vis[0][None]
    vis[4, :, :32] = 0
    xy = tr["xy"] * vis.repeat(2, axis=2)
    bt = gpu_pkg.EKFBatch(B, n)
    for t in range(T):
        off, ids, pts = _marker_list_with_strays(xy[t], vis[t], n, t)
        bt.step_known_sparse(np.ascontiguousarray(tr["twists"][t]), off, ids, pts)
    bt.sync()
    assert bt.update_count == int(vis.sum())
    states = bt.states()
    listed = dict(tr, xy=xy, vis=vis)
    for b in range(B):
        o = single.run_known(OracleEKF(n), listed, b)
        assert state_err(states[b], o.state) < TOL, b
        assert sigma_err(bt.sigma(b), o.sigma) < TOL, b


def _unknown_world(pkg):
    """49 tubes on a 7 x 7 grid, all within sight: more than 32 readings per step, and more tubes than slots for
    n < 49 (the map fills up and unmatched readings are dropped)."""
    return pkg.tracegen.grid_world(7, 7, pitch=0.45, max_visible=3.0)


@pytest.mark.parametrize("n,m_max", [(6, 1), (6, 7), (6, 40), (33, 1), (33, 7), (33, 40), (64, 1), (64, 7), (64, 40),
                                     (20, 40)])
def test_unknown_association_matches_oracle(gpu_pkg, n, m_max):
    """n = 20 runs the tile kernel, every other n the staircase kernel."""
    B, T = 6, 12
    w = _unknown_world(gpu_pkg)
    w.n_slots = n
    tu = gpu_pkg.tracegen.simulate_unknown(w, B, T, seed=500 + n + m_max, m_max=m_max)
    bt = gpu_pkg.EKFBatch(B, n)
    assoc = run_unknown(bt, tu, m_max)
    states, known = bt.states(), bt.known
    assert int(tu["count"].max()) == min(m_max, 49)
    created = full = 0
    for b in range(B):
        o = OracleEKF(n)
        k = np.zeros(n, np.uint8)
        for t, (a, dmin, sec, cr) in enumerate(single.run_unknown(o, tu, k, b)):
            m = len(a)
            assert_clear(dmin, sec)
            assert np.array_equal(assoc[t][b, :m], a), (b, t)
            assert np.all(assoc[t][b, m:] == -1)
            created += int(cr.sum())
            full += int(np.sum((dmin >= 10.0) & (cr == 0)))
        assert np.array_equal(known[b], k), b
        assert state_err(states[b], o.state) < TOL, b
        assert sigma_err(bt.sigma(b), o.sigma) < TOL, b
    assert created >= B * min(n, 5)
    if n == 6 or (n < 49 and m_max == 40):
        assert full > 0  # readings dropped because the map was full


@pytest.mark.parametrize("mode", ["known", "unknown"])
def test_checkpoint_resume_is_bit_identical(gpu_pkg, tmp_path, mode):
    n, B, T, M = 33, 24, 12, 40
    tr = _known_trace(gpu_pkg, n, B, T, seed=21)
    w = _unknown_world(gpu_pkg)
    w.n_slots = n
    tu = gpu_pkg.tracegen.simulate_unknown(w, B, T, seed=22, m_max=M)
    a, b = gpu_pkg.EKFBatch(B, n), gpu_pkg.EKFBatch(B, n)

    def step(bt, t):
        if mode == "known":
            step_known(gpu_pkg, bt, tr, t)
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
    for f in (0, B - 1):
        assert np.array_equal(a.sigma(f), b.sigma(f))
    assert a.update_count == b.update_count


def test_association_ties_lowest_index_wins(gpu_pkg):
    """Landmark i duplicated into slot j (state, Sigma rows and columns) through checkpoint() / restore(): a reading of
    that landmark is exactly as far from both, and the lower index must win.  (3, 9) sit in different lanes and meet in
    the shuffle merge; (5, 37) share lane 5, which scans both."""
    n, B = 64, 2
    N = 3 + 2 * n
    tr = _known_trace(gpu_pkg, n, B, 4, seed=31)
    bt = gpu_pkg.EKFBatch(B, n)
    run_known(gpu_pkg, bt, tr)
    ck = bt.checkpoint()
    ss, sts = stair_strides(N)
    size = stair_row_base(N, N)
    pairs = [(3, 9), (5, 37)]
    oracles = []
    for b, (i, j) in enumerate(pairs):
        dense = bt.sigma(b)
        assert np.array_equal(pack_staircase(dense, N), ck["sigma_packed"][b * ss:b * ss + size])
        st = ck["state"][b * sts:b * sts + N].copy()
        for src, dst in ((3 + 2 * i, 3 + 2 * j), (4 + 2 * i, 4 + 2 * j)):
            dense[dst, :] = dense[src, :]
            st[dst] = st[src]
        for src, dst in ((3 + 2 * i, 3 + 2 * j), (4 + 2 * i, 4 + 2 * j)):
            dense[:, dst] = dense[:, src]
        ck["sigma_packed"][b * ss:b * ss + size] = pack_staircase(dense, N)
        ck["state"][b * sts:b * sts + N] = st
        o = OracleEKF(n)
        o.state, o.sigma = st, dense
        oracles.append(o)
    ck["known"][:] = 1
    bt.restore(ck)
    tw = np.array([[0.02, 0.01], [-0.015, 0.02]])
    meas = np.zeros((B, 1, 2))
    for b, (i, j) in enumerate(pairs):
        oracles[b].prediction(*tw[b])
        meas[b, 0] = robot_frame(oracles[b].state, i, (0.01, -0.005))
    assoc = bt.step_unknown(tw, meas, np.ones(B, np.int32), 1, want_assoc=True)
    states = bt.states()
    for b, (i, j) in enumerate(pairs):
        k = np.ones(n, np.uint8)
        a, dmin, sec, cr = oracles[b].data_association(meas[b], k)
        assert a[0] == i and sec[0] == dmin[0] < 1.0  # the fixture is an exact tie on the oracle too
        assert assoc[b, 0] == i, (b, assoc[b])
        assert state_err(states[b], oracles[b].state) < TOL
        assert sigma_err(bt.sigma(b), oracles[b].sigma) < TOL


# ---------------------------------------------------------------- measurement counts outside [0, m_max]
def _count_fixture(pkg, n, B, M):
    """Two steps of M readings of the same M tubes per filter: the first creates the landmarks, the second updates
    them."""
    w = pkg.tracegen.default_world(n)
    w.max_visible = 3.0
    tu = pkg.tracegen.simulate_unknown(w, B, 2, seed=40 + n, m_max=M, shuffle=False)
    assert np.all(tu["count"] == M)
    return tu


@pytest.mark.parametrize("n", [20, 33])
def test_measurement_count_is_clamped(gpu_pkg, n):
    """ekf_batch_step_unknown(_dev): a count below 0 is an empty list (prediction only, outputs all -1, known list
    unchanged), a count above m_max is m_max, and a null count array means m_max for every filter.  n = 20 runs the
    tile kernel, n = 33 the staircase kernel."""
    import torch
    B, M = 8, 6
    tu = _count_fixture(gpu_pkg, n, B, M)
    tw0, tw1 = np.ascontiguousarray(tu["twists"][0]), np.ascontiguousarray(tu["twists"][1])
    me0, me1 = np.ascontiguousarray(tu["meas"][0]), np.ascontiguousarray(tu["meas"][1])
    full = np.full(B, M, np.int32)
    bad = full.copy()
    bad[3], bad[5] = -2, M + 5

    def batch():
        bt = gpu_pkg.EKFBatch(B, n)
        bt.step_unknown(tw0, me0, full, M)
        return bt

    # host path, filter 3 empty, filter 5 over-long
    a = batch()
    known0 = a.known
    assoc = a.step_unknown(tw1, me1, bad, M, want_assoc=True)
    states, known = a.states(), a.known
    for b in range(B):  # by hand: filter 3's second step is a prediction only
        o = OracleEKF(n)
        k = np.zeros(n, np.uint8)
        o.prediction(*tu["twists"][0, b])
        o.data_association(tu["meas"][0, b], k)
        o.prediction(*tu["twists"][1, b])
        if b == 3:
            assert np.all(assoc[b] == -1) and np.array_equal(known[b], known0[b])
        else:
            want, dmin, sec, _ = o.data_association(tu["meas"][1, b], k)
            assert_clear(dmin, sec)
            assert np.array_equal(assoc[b], want), (b, assoc[b], want)
            assert np.array_equal(known[b], k)
            if b == 2:
                assert np.all(want[4:] >= 0)  # readings 4 and 5 are real updates
        assert state_err(states[b], o.state) < TOL and sigma_err(a.sigma(b), o.sigma) < TOL, b

    # device pointers, the outputs preceded by a guard row: filter 0 is empty as well, and nothing may be written
    # before its outputs
    d = batch()
    bad_d = bad.copy()
    bad_d[0] = -3
    out = torch.full((B + 1, M), 77, dtype=torch.int32, device="cuda")
    t_tw, t_me, t_ct = dev(tw1), dev(me1), dev(bad_d)
    torch.cuda.synchronize()
    d.step_unknown_dev(t_tw.data_ptr(), t_me.data_ptr(), t_ct.data_ptr(), M, out[1].data_ptr())
    d.sync()
    got = out.cpu().numpy()
    assert np.all(got[0] == 77)
    assert np.all(got[1] == -1) and np.array_equal(got[2:], assoc[1:])
    assert np.array_equal(d.states()[1:], states[1:]) and np.array_equal(d.known[1:], known[1:])
    o = OracleEKF(n)
    o.prediction(*tu["twists"][0, 0])
    o.data_association(tu["meas"][0, 0], np.zeros(n, np.uint8))
    o.prediction(*tu["twists"][1, 0])
    assert state_err(d.states()[0], o.state) < TOL and sigma_err(d.sigma(0), o.sigma) < TOL
    assert np.array_equal(d.known[0], known0[0])

    # no count array: m_max readings for every filter, bit-identical to the host path with count = m_max
    e, f = batch(), batch()
    out_e = torch.zeros((B, M), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    e.step_unknown_dev(t_tw.data_ptr(), t_me.data_ptr(), None, M, out_e.data_ptr())
    e.sync()
    assoc_f = f.step_unknown(tw1, me1, full, M, want_assoc=True)
    assert np.array_equal(out_e.cpu().numpy(), assoc_f)
    assert np.array_equal(e.states(), f.states()) and np.array_equal(e.known, f.known)
    for b in (0, B - 1):
        assert np.array_equal(e.sigma(b), f.sigma(b))
