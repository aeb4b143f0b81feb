"""Host side of the consistency read-out: chi-square bounds, ANEES from the batch partial, and the report's table."""
import numpy as np
import pytest


@pytest.mark.parametrize("dof", [2, 3])
@pytest.mark.parametrize("runs", [15, 16, 64, 1000, 4096, 65536])
@pytest.mark.parametrize("p", [0.95, 0.9])
def test_chi2_bounds_match_scipy(pkg, dof, runs, p):
    from scipy.stats import chi2
    k = dof * runs
    assert k >= 30
    lo, hi = pkg.consistency.chi2_bounds(dof, runs, p)
    np.testing.assert_allclose(lo, chi2.ppf((1 - p) / 2, k) / runs, rtol=1e-3)
    np.testing.assert_allclose(hi, chi2.ppf((1 + p) / 2, k) / runs, rtol=1e-3)
    assert lo < dof < hi


def test_product_package_does_not_import_scipy(pkg):
    import inspect
    assert "scipy" not in inspect.getsource(pkg.consistency)


def test_anees_from_stats(pkg):
    pose = np.array([2.0, 4.0, 3.0])
    lm = np.array([1.0, 0.5, 2.5, 4.0])
    s = [pose.sum(), (pose ** 2).sum(), 3, lm.sum(), (lm ** 2).sum(), 4, 1, 2]
    c = pkg.consistency.anees_from_stats(s)
    assert c["pose_anees"] == pytest.approx(3.0) and c["pose_nees_var"] == pytest.approx(pose.var())
    assert c["landmark_anees"] == pytest.approx(2.0) and c["landmark_nees_var"] == pytest.approx(lm.var())
    assert (c["pose_count"], c["landmark_count"], c["pose_singular"], c["landmark_singular"]) == (3, 4, 1, 2)
    # partials of two ranks add up to the partial of the whole batch
    half = pkg.consistency.anees_from_stats(np.add(s, s))
    assert half["pose_anees"] == pytest.approx(3.0) and half["pose_count"] == 6
    empty = pkg.consistency.anees_from_stats(np.zeros(8))
    assert np.isnan(empty["pose_anees"]) and np.isnan(empty["landmark_anees"])


def test_report_renders_the_consistency_table(pkg):
    r = {"robots": 2, "steps": 3, "seed": 0, "updates": 11, "landmark_rmse": 0.01, "landmarks": 20,
         "rmse_xytheta": {"slam": [0.001, 0.002, 0.01], "prediction_only": [0.1, 0.2, 0.3], "wheel_odometry": [0, 0, 0]},
         "worst_xy_error": {"slam": 0.004, "prediction_only": 0.3, "wheel_odometry": 0.0}}
    row = {"anees": 3.5, "dof": 3, "runs": 2, "singular": 0, "bounds_95": [0.8, 6.2]}
    r["consistency"] = {"slam": {"pose": row, "landmarks": dict(row, dof=2, anees=1.25, runs=40)},
                        "prediction_only": {"pose": dict(row, anees=12.0)},
                        "pose_anees_series": {"steps": [1, 2, 3], "anees": [1.0, 2.0, 3.5]}}
    md = pkg.report.markdown(r)
    assert "Slam | 0.00100 | 0.00200" in md
    assert "Slam | pose | 3 | 3.500 | 0.800 .. 6.200 | 2 | 0" in md
    assert "Slam | landmarks | 2 | 1.250 |" in md and "Prediction only | pose | 3 | 12.000 |" in md
    assert "3: 3.500" in md
