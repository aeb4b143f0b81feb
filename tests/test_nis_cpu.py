"""Host side of the batch NIS read-out: consistency.anis_from_stats, the report's innovations row, and the NIS of
tests/_noise_ref.py (the numpy restatement of the CPU oracle) against nu^T S^-1 nu formed directly from its sigma and
state."""
import math

import numpy as np
import pytest

from _noise_ref import NoiseOracle, normalize_angle


def test_anis_from_stats_and_bounds(pkg):
    cs = pkg.consistency
    r = cs.anis_from_stats([10.0, 60.0, 5.0, 2.0])
    assert r["anis"] == 2.0 and r["nis_var"] == 60.0 / 5 - 4.0 and r["count"] == 5 and r["nonfinite"] == 2
    assert r["dof"] == 2 and r["bounds_95"] == cs.chi2_bounds(2, 5)
    lo, hi = cs.anis_from_stats([0, 0, 1000, 0])["bounds_95"]
    assert lo < 2.0 < hi
    e = cs.anis_from_stats(np.zeros(4))
    assert math.isnan(e["anis"]) and math.isnan(e["nis_var"]) and e["count"] == 0
    with pytest.raises(ValueError):
        cs.anis_from_stats([1.0, 2.0, 3.0])


def _direct_nis(state, sigma, i, sx, sy):
    """nu^T S^-1 nu of landmark i at the state's pose, from the dense H_j"""
    th, x, y = state[:3]
    mx, my = state[3 + 2 * i], state[4 + 2 * i]
    dx, dy = mx - x, my - y
    d = dx * dx + dy * dy
    q = math.sqrt(d)
    H = np.zeros((2, len(state)))
    H[0, [1, 2, 3 + 2 * i, 4 + 2 * i]] = [-dx / q, -dy / q, dx / q, dy / q]
    H[1, [0, 1, 2, 3 + 2 * i, 4 + 2 * i]] = [-1.0, dy / d, -dx / d, -dy / d, dx / d]
    S = H @ sigma @ H.T + 0.01 * np.eye(2)
    zphi = normalize_angle(math.atan2(dy, dx) - th)
    nu = np.array([math.hypot(sx, sy) - q, normalize_angle(math.atan2(sy, sx) - zphi)])
    return float(nu @ np.linalg.solve(S, nu))


@pytest.fixture(scope="module")
def one_landmark_trace(pkg):
    """A trace that sees exactly one landmark per step (after a first call that lists them all)."""
    tg = pkg.tracegen
    tr = tg.simulate_known(tg.grid_world(5, 4, pitch=0.35), 1, 12, seed=5)
    vis = np.zeros((12, 20), np.uint8)
    vis[0] = 1
    for t in range(1, 12):
        vis[t, (3 * t) % 20] = 1
    return tr["twists"][:, 0], tr["xy"][:, 0], vis


def test_reference_nis_matches_direct_formula(one_landmark_trace):
    tw, xy, vis = one_landmark_trace
    o = NoiseOracle(20)
    for t in range(len(tw)):
        o.prediction(*tw[t])
        st, sig = o.state.copy(), o.sigma.copy()
        before = len(o.values)
        o.measurement(xy[t], vis[t])
        if t == 0:
            assert len(o.values) == 0  # the first call's landmarks start at their readings: not scored
            continue
        i = int(np.flatnonzero(vis[t])[0])
        want = _direct_nis(st, sig, i, xy[t, 2 * i], xy[t, 2 * i + 1])
        assert len(o.values) == before + 1
        assert o.values[-1] == pytest.approx(want, rel=1e-9)
    assert o.acc[2] == len(tw) - 1 and o.acc[3] == 0
    assert o.acc[0] == pytest.approx(sum(o.values), rel=1e-14)
    assert o.acc[1] == pytest.approx(sum(v * v for v in o.values), rel=1e-14)


def test_reference_scoring_rule_on_the_association_path():
    o = NoiseOracle(20)
    known = np.zeros(20, np.uint8)
    o.prediction(0.01, 0.05)
    a, c = o.data_association(np.array([[1.0, 0.2]]), known)
    assert a[0] == 0 and c[0] == 1 and o.acc[2] == 0  # created by this reading: corrected, not scored
    o.prediction(0.01, 0.05)
    a, c = o.data_association(np.array([[0.95, 0.2]]), known)
    assert a[0] == 0 and c[0] == 0 and o.acc[2] == 1  # the same landmark again: scored


def test_report_renders_the_innovations_row(pkg):
    r = {"robots": 2, "steps": 3, "seed": 0, "updates": 11, "landmark_rmse": 0.01, "landmarks": 20,
         "rmse_xytheta": {"slam": [0.001, 0.002, 0.01], "prediction_only": [0.1, 0.2, 0.3], "wheel_odometry": [0, 0, 0]},
         "worst_xy_error": {"slam": 0.004, "prediction_only": 0.3, "wheel_odometry": 0.0}}
    row = {"anees": 3.5, "dof": 3, "runs": 2, "singular": 0, "bounds_95": [0.8, 6.2]}
    r["consistency"] = {"slam": {"pose": row, "landmarks": dict(row, dof=2, anees=1.25, runs=40)},
                        "prediction_only": {"pose": dict(row, anees=12.0)}}
    assert "innovations" not in pkg.report.markdown(r)
    r["consistency"]["slam"]["innovations"] = {"anis": 2.25, "dof": 2, "bounds_95": [1.9, 2.1], "corrections": 900,
                                               "nonfinite": 0}
    md = pkg.report.markdown(r)
    assert "Slam | innovations | 2 | 2.250 | 1.900 .. 2.100 | 900 | 0" in md
    assert "Slam | pose | 3 | 3.500 | 0.800 .. 6.200 | 2 | 0" in md
