"""Host side of per-filter noise: the noise-aware reference of tests/_noise_ref.py against the CPU oracle and a
closed form, and the Python packing of noise rows."""
import math

import numpy as np
import pytest

from _noise_ref import NoiseOracle
from _oracle import OracleEKF


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def test_reference_values_are_bit_identical_to_the_oracle(pkg):
    """With the reference values set explicitly the noise-aware reference is the oracle, bit for bit, over a known
    and an unknown association trace."""
    tg = pkg.tracegen
    n, T = 20, 12
    tr = tg.simulate_known(tg.grid_world(5, 4, pitch=0.35), 1, T, seed=3)
    o, r = OracleEKF(n), NoiseOracle(n, (1e-4, 1e-4, 1e-4, 0.01, 0.01))
    for t in range(T):
        o.prediction(*tr["twists"][t, 0])
        r.prediction(*tr["twists"][t, 0])
        o.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        r.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        assert _same(o.state, r.state) and _same(o.sigma, r.sigma), t
    tu = tg.simulate_unknown(tg.dense_world(n), 1, T, seed=4, m_max=40)
    o, r = OracleEKF(n), NoiseOracle(n)
    ko, kr = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for t in range(T):
        o.prediction(*tu["twists"][t, 0])
        r.prediction(*tu["twists"][t, 0])
        m = int(tu["count"][t, 0])
        a_o, _, _, c_o = o.data_association(tu["meas"][t, 0, :m], ko)
        a_r, c_r = r.data_association(tu["meas"][t, 0, :m], kr)
        assert np.array_equal(a_o, a_r) and np.array_equal(c_o, c_r) and np.array_equal(ko, kr), t
        assert _same(o.state, r.state) and _same(o.sigma, r.sigma), t


def _dense_h(state, i):
    th, x, y = state[:3]
    dx, dy = state[3 + 2 * i] - x, state[4 + 2 * i] - y
    d = dx * dx + dy * dy
    q = math.sqrt(d)
    H = np.zeros((2, len(state)))
    H[0, [1, 2, 3 + 2 * i, 4 + 2 * i]] = [-dx / q, -dy / q, dx / q, dy / q]
    H[1, [0, 1, 2, 3 + 2 * i, 4 + 2 * i]] = [-1.0, dy / d, -dx / d, -dy / d, dx / d]
    return H, q, math.atan2(dy, dx) - th


def test_scaled_r_matches_closed_form(pkg):
    """With R scaled, S = H Sigma H^T + R and the Mahalanobis distance (bearing not wrapped) match numpy."""
    tg = pkg.tracegen
    n = 20
    tr = tg.simulate_known(tg.grid_world(5, 4, pitch=0.35), 1, 6, seed=9)
    noise = (3e-4, 2e-4, 5e-5, 0.004, 0.0025)
    r = NoiseOracle(n, noise)
    for t in range(6):
        r.prediction(*tr["twists"][t, 0])
        r.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
    R = np.diag(noise[3:])
    rng = np.random.default_rng(0)
    for i in range(n):
        H, zr, zphi = _dense_h(r.state, i)
        S = H @ r.sigma @ H.T + R
        got, _, _ = r.innovation_covariance(i, *r.state[:3])
        assert np.allclose(np.array(got), S, rtol=1e-10, atol=1e-14)
        sx, sy = rng.normal(0, 1.0, 2)
        nu = np.array([math.hypot(sx, sy) - zr, math.atan2(sy, sx) - math.atan2(math.sin(zphi), math.cos(zphi))])
        want = float(nu @ np.linalg.solve(S, nu))
        assert math.isclose(r.maha(sx, sy, i), want, rel_tol=1e-9), i


def test_noise_rows_broadcast_and_shapes(pkg):
    rows = pkg.ekf_slam.noise_rows
    one = rows([1, 2, 3], [4, 5], 7)
    assert one.shape == (1, 5) and one.tolist() == [[1, 2, 3, 4, 5]]
    assert rows(None, None, 3).tolist() == [[1e-4, 1e-4, 1e-4, 0.01, 0.01]]
    per = rows(np.arange(9.0).reshape(3, 3), [0.5, 0.25], 3)
    assert per.shape == (3, 5) and np.all(per[:, 3:] == [0.5, 0.25]) and np.array_equal(per[:, :3], np.arange(9.0).reshape(3, 3))
    with pytest.raises(ValueError):
        rows([1, 2], None, 3)
    with pytest.raises(ValueError):
        rows(None, np.ones((2, 2)), 3)
