"""Helpers shared by the GPU batch tests: device shorthands, the grid world and traces the batch tests run, the step
loops over EKFBatch's input forms, the bit-identity checks of checkpoints and replicas, the association tie margin and
the staircase layout's strides.  What differs between test files (number of trajectories, m_max, tolerances) is
passed in."""
import numpy as np


def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def c(a):
    return np.ascontiguousarray(a)


def grid_world(pkg, n):
    nx = max(d for d in range(1, int(np.sqrt(n)) + 1) if n % d == 0)  # n landmarks on an nx x (n / nx) grid
    return pkg.tracegen.grid_world(n // nx, nx, pitch=0.35)


def known_trace(pkg, n, B, T, seed, p_vis=0.5):
    """The simulator's trace with each visible reading kept at probability p_vis; the first call lists every slot, so
    that each landmark starts at its reading (and every slot takes a correction that is not scored)."""
    tr = pkg.tracegen.simulate_known(grid_world(pkg, n), B, T, seed=seed)
    rng = np.random.default_rng(seed)
    vis = (tr["vis"] != 0) & (rng.random(tr["vis"].shape) < p_vis)
    vis[0] = True
    vis = vis.astype(np.uint8)
    return {"twists": tr["twists"], "xy": np.ascontiguousarray(tr["xy"] * vis.repeat(2, axis=2)), "vis": vis}


def unknown_trace(pkg, n, B, T, seed, m_max):
    return pkg.tracegen.simulate_unknown(pkg.tracegen.dense_world(n), B, T, seed=seed, m_max=m_max)


def step_known(pkg, bt, tr, t, form="dense"):
    """Step t of a known-association trace as dense host arrays, a marker list, or dense device arrays."""
    tw, xy, vis = c(tr["twists"][t]), c(tr["xy"][t]), c(tr["vis"][t])
    if form == "dense":
        bt.step_known(tw, xy, vis)
    elif form == "markers":
        bt.step_known_sparse(tw, *pkg.marker_list(xy, vis))
    else:
        d = (dev(tw), dev(xy), dev(vis))
        bt.step_known_dev(*(x.data_ptr() for x in d))
        bt.sync()  # the tensors may go once the step has read them


def run_known(pkg, bt, tr, form="dense"):
    for t in range(tr["twists"].shape[0]):
        step_known(pkg, bt, tr, t, form)
    bt.sync()


def run_unknown(bt, tr, m_max):
    """Every step of an unknown-association trace; returns the association outputs [T, B, m_max]."""
    out = [bt.step_unknown(c(tr["twists"][t]), c(tr["meas"][t]), c(tr["count"][t]), m_max, want_assoc=True)
           for t in range(tr["twists"].shape[0])]
    bt.sync()
    return np.stack(out)


def assert_same_checkpoint(a, b):
    for key in ("sigma_packed", "state", "init_flag", "known"):
        x, y = a[key], b[key]
        if x.dtype == np.float64:
            x, y = x.view(np.uint64), y.view(np.uint64)
        assert np.array_equal(x, y), key
    assert a["updates"] == b["updates"]


def replicate(a, B, K):
    """[T, K, ...] -> [T, B, ...]: filter b runs trajectory b mod K."""
    return np.ascontiguousarray(a[:, np.arange(B) % K])


def assert_replicas(a, B, K, what):
    """Rows b and b mod K of a [B, ...] array are bit-identical (floats compared as their bit patterns)."""
    a = np.ascontiguousarray(a).reshape(B, -1)
    if a.dtype == np.float64:
        a = a.view(np.uint64)
    for k in range(K):
        bad = np.flatnonzero((a[k::K] != a[k]).any(axis=1))
        assert bad.size == 0, f"{what}: filter {k + K * int(bad[0])} differs from filter {k}"


def tie_margin(dmin, second):
    """How far each association decision is from flipping: dmin's distance to the gates (1 and 10) and to the
    runner-up, or, when no candidate is below the gate (dmin == 10 exactly), the runner-up's distance to the gate."""
    has = dmin < 10.0
    return np.where(has, np.minimum.reduce([np.abs(dmin - 10.0), np.abs(dmin - 1.0), np.abs(second - dmin)]),
                    np.abs(second - 10.0))


def assert_clear(dmin, second):
    """No decision sits within 1e-6 (relative) of a gate or of a tie with the runner-up, where the device and the
    oracle could round to different sides."""
    margin = tie_margin(dmin, second)
    assert np.all(margin > 1e-6 * np.maximum(1.0, np.abs(dmin))), "threshold tie in the fixture: pick another seed"


def stair_row_base(r, N):
    """Offset of row r in the packed staircase layout of csrc/ekf_fused_sym.cuh (the batch layout of n <= 64, n != 20):
    row r keeps the columns [16 floor(r / 16), N)."""
    rb = r >> 4
    return 16 * rb * N - 128 * rb * (rb - 1) + (r - 16 * rb) * (N - 16 * rb)


def stair_strides(N):
    return (stair_row_base(N, N) + 1) & ~1, (N + 1) & ~1  # per-filter Sigma and state strides in doubles


def robot_frame(state, k, offset=(0.0, 0.0)):
    """Reading of landmark k's current estimate as the robot sees it from the estimated pose, plus an offset."""
    th, x, y = state[:3]
    dx, dy = state[3 + 2 * k] - x, state[4 + 2 * k] - y
    c, s = np.cos(th), np.sin(th)
    return np.array([c * dx + s * dy + offset[0], -s * dx + c * dy + offset[1]])
