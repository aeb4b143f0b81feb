"""Filter consistency statistics on the host side of EKFBatch.nees() / nees_dev() and nis() / nis_dev() (numpy and the
standard library only).

A consistent filter's NEES (normalised estimation error squared, e^T P^-1 e) is chi-square distributed with as many
degrees of freedom as the block it scores: 3 for the pose, 2 for a landmark.  Averaged over `runs` independent
Monte-Carlo runs (ANEES), runs * ANEES is chi-square with dof * runs degrees of freedom, so a consistent filter's ANEES
lies inside chi2_bounds(dof, runs) with probability p; an ANEES above the interval means an overconfident covariance.

The batch partial of ekf_batch_nees, out8 = {sum NEES_pose, sum NEES_pose^2, #pose, sum NEES_lm, sum NEES_lm^2, #lm,
#singular pose, #singular lm}, is additive: a multi-GPU run sums the ranks' vectors with sharding.allreduce_sum and
passes the sum to anees_from_stats.

NIS (normalised innovation squared, nu^T S^-1 nu of one range-bearing correction) needs no truth and is chi-square with
2 degrees of freedom for a consistent filter.  The batch total of EKFBatch.nis() / ekf_batch_nis, out4 = {sum NIS,
sum NIS^2, #scored, #non-finite}, is additive in the same way; anis_from_stats gives the ANIS and its interval."""
from statistics import NormalDist

import numpy as np


def anees_from_stats(out8):
    """out8 (one batch, or the sum over batches or ranks) -> dict of ANEES, their sample variances, and counts."""
    s = np.asarray(out8, dtype=np.float64).reshape(8)

    def mean_var(total, squares, count):
        if count <= 0:
            return float("nan"), float("nan")
        m = total / count
        return float(m), float(squares / count - m * m)

    pm, pv = mean_var(s[0], s[1], s[2])
    lm, lv = mean_var(s[3], s[4], s[5])
    return {"pose_anees": pm, "pose_nees_var": pv, "pose_count": int(s[2]), "pose_singular": int(s[6]),
            "landmark_anees": lm, "landmark_nees_var": lv, "landmark_count": int(s[5]), "landmark_singular": int(s[7])}


def anis_from_stats(out4):
    """NIS partial of EKFBatch.nis() / ekf_batch_nis, out4 = {sum NIS, sum NIS^2, #scored, #non-finite} (one batch, or
    the sum over batches or ranks) -> ANIS, its sample variance, the counts, and the 95 % interval of a consistent
    filter's ANIS over that many corrections (the NIS of one range-bearing correction is chi-square with 2 degrees of
    freedom)."""
    s = np.asarray(out4, dtype=np.float64).reshape(4)
    count = int(s[2])
    if count > 0:
        m = s[0] / count
        mean, var = float(m), float(s[1] / count - m * m)
    else:
        mean = var = float("nan")
    return {"anis": mean, "nis_var": var, "count": count, "nonfinite": int(s[3]), "dof": 2,
            "bounds_95": chi2_bounds(2, count)}


def chi2_quantile(q, k):
    """q-quantile of chi-square with k degrees of freedom, Wilson-Hilferty approximation (relative error below 1e-3
    for k >= 30 at the 95 % two-sided quantiles)."""
    z = NormalDist().inv_cdf(q)
    h = 2.0 / (9.0 * k)
    return k * (1.0 - h + z * np.sqrt(h)) ** 3


def chi2_bounds(dof, runs, p=0.95):
    """Two-sided probability-p interval of the ANEES of a consistent filter over `runs` runs of a dof-dimensional
    block: chi2((1 -+ p) / 2, dof * runs) / runs."""
    k = float(dof) * float(runs)
    if k <= 0:
        return float("nan"), float("nan")
    return float(chi2_quantile((1.0 - p) / 2.0, k) / runs), float(chi2_quantile((1.0 + p) / 2.0, k) / runs)
