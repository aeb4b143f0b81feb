"""Helpers shared by the GPU single-filter tests: the engine names, and one replay of trajectory b of a batch trace
through a device filter (EKF_SLAM, ShardedEKF) or a CPU reference (OracleEKF, NoiseOracle).  One step is prediction()
then measurement() on a known-association trace, or prediction() then data_association() on the first count[t, b]
readings of an unknown-association one."""
import numpy as np

from _batch import grid_world, known_trace, unknown_trace
from _noise_ref import NoiseOracle
from _oracle import OracleEKF, sigma_err, state_err


def engine(pkg, name):
    return pkg.ENGINE_FUSED if name == "fused" else pkg.ENGINE_STREAM


def bits(a):
    """A float64 array as its bit patterns, for bit-for-bit comparisons."""
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def sigma(f):
    return f.sigma_full_local() if hasattr(f, "sigma_full_local") else f.sigma


def _predict(f, twist):
    if isinstance(f, (OracleEKF, NoiseOracle)):
        f.prediction(*twist)  # the references take (dtheta, dx) as two arguments, the device filters as a pair
    else:
        f.prediction(tuple(twist))


def step_known(f, tr, t, b=0):
    _predict(f, tr["twists"][t, b])
    f.measurement(tr["xy"][t, b], tr["vis"][t, b])


def step_unknown(f, tr, t, known, b=0):
    """Returns what f.data_association returns: a dict on a device filter, a tuple on a reference.  The reading count is
    clamped to [0, m_max] as the batch engines clamp it."""
    _predict(f, tr["twists"][t, b])
    m = min(max(int(tr["count"][t, b]), 0), tr["meas"].shape[2])
    return f.data_association(tr["meas"][t, b, :m], known)


def run_known(f, tr, b=0, steps=None):
    """Steps `steps` (default: all) of trajectory b through f; returns f."""
    for t in range(tr["twists"].shape[0]) if steps is None else steps:
        step_known(f, tr, t, b)
    return f


def run_unknown(f, tr, known, b=0, steps=None):
    """Steps `steps` (default: all) of trajectory b through f; returns the data_association outputs, one per step."""
    return [step_unknown(f, tr, t, known, b) for t in (range(tr["twists"].shape[0]) if steps is None else steps)]


def streamed(pkg, n, tr, b, steps):
    """Trajectory b through a streamed filter whose pending corrections do not outlive a call, as in a wide batch."""
    f = pkg.EKF_SLAM(n, engine=pkg.ENGINE_STREAM)
    f.set_carry_pending(False)
    return run_known(f, tr, b, steps)


def parity_known(f, o, tr, check_every=1):
    """Trajectory 0 through the device filter f and the reference o; the worst state and Sigma errors, read after
    every check_every-th step and after the last."""
    worst_x = worst_s = 0.0
    T = tr["twists"].shape[0]
    for t in range(T):
        step_known(f, tr, t)
        step_known(o, tr, t)
        if t % check_every == 0 or t == T - 1:
            worst_x = max(worst_x, state_err(f.state, o.state))
            worst_s = max(worst_s, sigma_err(sigma(f), o.sigma))
    return worst_x, worst_s


def traces(pkg, n, T, seed, m_max):
    """A known-association trace and an unknown-association one (seed + 1) for one filter."""
    if n <= 33:
        tu = unknown_trace(pkg, n, 1, T, seed=seed + 1, m_max=m_max)
    else:  # the dense world holds about 33 tubes; larger maps take the grid of the known traces
        tu = pkg.tracegen.simulate_unknown(grid_world(pkg, n), 1, T, seed=seed + 1, m_max=m_max)
    return known_trace(pkg, n, 1, T, seed), tu


def nis_step_known(o, tr, t, b=0):
    """Step t through the NoiseOracle o; returns the last_nis() a filter should give for it: n values, -1 where nothing
    was scored (every slot of the first measurement(), the slots not visible)."""
    k0, score = len(o.values), o.init_flag
    step_known(o, tr, t, b)
    want = np.full(o.n, -1.0)
    if score:
        want[np.flatnonzero(tr["vis"][t, b])] = o.values[k0:]
    return want


def nis_step_unknown(o, tr, t, known, b=0):
    """As nis_step_known for an unknown-association step: m values, -1 for a reading that was dropped or created its
    landmark.  Returns (assoc, created, expected last_nis())."""
    k0 = len(o.values)
    a, cr = step_unknown(o, tr, t, known, b)
    want = np.full(len(a), -1.0)
    want[(a >= 0) & (cr == 0)] = o.values[k0:]
    return a, cr, want
