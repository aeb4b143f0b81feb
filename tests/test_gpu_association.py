"""The association argmin of the single-filter engines where it has something to merge, against the CPU oracle.

Each engine finds the nearest known landmark (Mahalanobis distance) and the runner-up in stages: per lane over the
landmarks the lane scans, then across the warp's lanes (fused engine, n > 32 gives a lane two landmarks), and for the
streamed and row-sharded engines across warps, across the ceil(known / 256) CTAs of the scan and across ranks.  The
map here is built with known association, then readings are aimed at chosen landmarks - the oracle's current estimate
of a landmark in the robot frame, plus an offset - so that the winner, the runner-up or a tie sits where two stages
meet.  Every output of every call is compared: association, created flag, distance, runner-up, known list, state and
covariance.  Ties must go to the lower index with runner-up == distance, and a NaN distance never wins."""
import functools

import numpy as np
import pytest

from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu

TOL = 1e-9
FAR = np.array([40.0, 35.0])  # a reading far from every landmark: a new one, or dropped when the map is full


def _robot_frame(state, k, offset=(0.0, 0.0)):
    """Reading of landmark k's current estimate as the robot sees it from the estimated pose, plus an offset."""
    th, x, y = state[:3]
    dx, dy = state[3 + 2 * k] - x, state[4 + 2 * k] - y
    c, s = np.cos(th), np.sin(th)
    return np.array([c * dx + s * dy + offset[0], -s * dx + c * dy + offset[1]])


@functools.lru_cache(maxsize=None)
def _map(n):
    """Known-association inputs that build an n-landmark map (0.45 m grid): the first call initialises every slot and
    corrects all of them, the second all again and the third every other one.  Returns the inputs and the oracle's
    result."""
    nx = int(np.ceil(np.sqrt(n)))
    i = np.arange(n)
    lm = np.stack([(i % nx - (nx - 1) / 2) * 0.45 + 0.13, (i // nx - (-(-n // nx) - 1) / 2) * 0.45 + 0.29], 1)
    rng = np.random.default_rng(n)
    o = OracleEKF(n)
    steps = []
    for tw, every in (((0.05, 0.02), 1), ((-0.03, 0.04), 1), ((0.02, -0.03), 2)):
        o.prediction(*tw)
        th, x, y = o.state[:3]
        d = lm - [x, y]
        c, s = np.cos(th), np.sin(th)
        xy = (np.stack([c * d[:, 0] + s * d[:, 1], -s * d[:, 0] + c * d[:, 1]], 1) + rng.normal(0, 0.005, d.shape)).ravel()
        vis = (i % every == 0).astype(np.uint8)
        o.measurement(xy, vis)
        steps.append((tw, xy, vis))
    return steps, o.state, o.sigma


def _sigma(f):
    return f.sigma_full_local() if hasattr(f, "sigma_full_local") else f.sigma


def _built(f, n):
    """Runs the map inputs through the device filter f; returns an oracle holding the same map."""
    steps, st, sg = _map(n)
    for tw, xy, vis in steps:
        f.prediction(tw)
        f.measurement(xy, vis)
    assert state_err(f.state, st) < TOL and sigma_err(_sigma(f), sg) < TOL
    o = OracleEKF(n)
    o.state, o.sigma, o.init_flag = st, sg, True
    return o


def _set(f, o, state, sigma):
    f.state, f.sigma = state, sigma
    o.state, o.sigma = state, sigma


def _duplicate(state, sigma, i, j, shift=(0.0, 0.0)):
    """Landmark i copied into slot j (state, Sigma rows and columns), then moved by `shift` (world frame)."""
    st, sg = state.copy(), sigma.copy()
    rows = ((3 + 2 * i, 3 + 2 * j), (4 + 2 * i, 4 + 2 * j))
    for src, dst in rows:
        sg[dst, :] = sg[src, :]
        st[dst] = st[src]
    for src, dst in rows:
        sg[:, dst] = sg[:, src]
    st[3 + 2 * j] += shift[0]
    st[4 + 2 * j] += shift[1]
    return st, sg


def _graze(o, k, known_count):
    """A reading moved away from landmark k until its nearest known landmark is at Mahalanobis distance 1.6: dropped.
    Of 24 directions the first in which that nearest landmark is k itself, else the first that gives a drop."""
    def nearest(xy):
        d = np.array([o.maha(*xy, i) for i in range(known_count)])
        return d.min(), int(np.argmin(d))

    first = None
    for ang in np.linspace(0.0, 2 * np.pi, 24, endpoint=False):
        u = np.array([np.cos(ang), np.sin(ang)])
        lo, hi = 0.0, 4.0
        for _ in range(40):
            mid = 0.5 * (lo + hi)
            lo, hi = (mid, hi) if nearest(_robot_frame(o.state, k, mid * u))[0] < 1.6 else (lo, mid)
        xy = _robot_frame(o.state, k, hi * u)
        d, i = nearest(xy)
        if d < 1.0:  # every point within reach in this direction is close to some landmark
            continue
        if i == k:
            return xy
        first = xy if first is None else first
    assert first is not None
    return first


def _assert_clear(dmin, second):
    """No decision sits within 1e-6 (relative) of a gate or of the runner-up, where the device and the oracle could
    round to different sides."""
    has = dmin < 10.0
    margin = np.where(has, np.minimum.reduce([np.abs(dmin - 10.0), np.abs(dmin - 1.0), np.abs(second - dmin)]),
                      np.abs(second - 10.0))
    assert np.all(margin > 1e-6 * np.maximum(1.0, np.abs(dmin))), "threshold tie in the fixture"


def _associate(f, o, xy, known_count, tie=False, nan_entry=None):
    """One data_association() call on the device filter and on the oracle with a known prefix of known_count ones;
    every output must agree.  Returns the oracle's (assoc, dmin, second, created)."""
    xy = np.asarray(xy, np.float64).reshape(-1, 2)
    kf = (np.arange(o.n) < known_count).astype(np.uint8)
    ko = kf.copy()
    r = f.data_association(xy, kf)
    a, dmin, sec, cr = o.data_association(xy, ko)
    if tie:
        assert np.all(sec == dmin) and np.all(r["second"] == r["dmin"])
    else:
        _assert_clear(dmin, sec)
    assert np.array_equal(r["assoc"], a), (r["assoc"], a)
    assert np.array_equal(r["created"], cr) and np.array_equal(kf, ko)
    np.testing.assert_allclose(r["dmin"], dmin, rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(r["second"], sec, rtol=1e-7, atol=1e-9)
    fs, os_ = f.state, o.state
    if nan_entry is not None:
        assert np.isnan(fs[nan_entry]) and np.isnan(os_[nan_entry])
        fs[nan_entry] = os_[nan_entry] = 0.0
    assert state_err(fs, os_) < TOL
    assert sigma_err(_sigma(f), o.sigma) < TOL
    return a, dmin, sec, cr


def _hit(f, o, k, partner, base):
    """A reading of landmark k, offset by `off`, with a copy of k moved by -3 `off` in slot `partner` as the runner-up."""
    off = np.array([0.01, -0.005])
    c, s = np.cos(base[0][0]), np.sin(base[0][0])
    _set(f, o, *_duplicate(*base, k, partner, shift=-3.0 * np.array([c * off[0] - s * off[1], s * off[0] + c * off[1]])))
    xy = _robot_frame(o.state, k, off)
    d_partner = o.maha(*xy, partner)
    a, dmin, sec, cr = _associate(f, o, xy, o.n)
    assert a[0] == k and cr[0] == 0 and sec[0] == d_partner


def _tie(f, o, i, j, base):
    """Landmark i copied into slot j: a reading of it is exactly as far from both, and the lower index wins."""
    _set(f, o, *_duplicate(*base, i, j))
    a, _, _, _ = _associate(f, o, _robot_frame(o.state, i, (0.01, -0.005)), o.n, tie=True)
    assert a[0] == min(i, j)


@pytest.mark.parametrize("n", [33, 48, 64])
def test_fused_single_filter(gpu_pkg, n):
    """One warp scans the map: lane l holds landmarks l and l + 32, merged by shuffles."""
    f = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_FUSED)
    o = _built(f, n)
    base = (o.state, o.sigma)
    for k in sorted({0, 31, 32, 33, n - 1} & set(range(n))):
        _hit(f, o, k, (k + 1) % n, base)  # the runner-up in the next lane
        _set(f, o, *base)
        a, _, _, cr = _associate(f, o, _graze(o, k, n), n)
        assert a[0] == -1 and cr[0] == 0
    for kc in (n // 2, n):  # a new landmark, then the full map drops the reading
        _set(f, o, *base)
        a, _, _, cr = _associate(f, o, FAR, kc)
        assert (a[0], cr[0]) == ((kc, 1) if kc < n else (-1, 0))
    i = {33: 0, 48: 9, 64: 29}[n]
    for p, q in ((i, i + 1), (i, i + 32), (i + 32, i + 1)):  # the last: a higher lane with the lower index wins
        _tie(f, o, p, q, base)


@pytest.mark.parametrize("max_pending", [1, None], ids=["pending1", "default"])
def test_streamed_engine(gpu_pkg, max_pending):
    """n = 600: three association CTAs of 256 landmarks, merged by the last CTA to finish.  The engine flushes its
    pending corrections before each distance, so the number it keeps pending must not matter."""
    n = 600
    f = gpu_pkg.EKF_SLAM(n, engine=gpu_pkg.ENGINE_STREAM)
    if max_pending:
        f.set_max_pending(max_pending)
    o = _built(f, n)
    base = (o.state, o.sigma)
    for k in (0, 255, 256, 511, 512, 599):
        _hit(f, o, k, k + 256 if k + 256 < n else k - 256, base)  # the runner-up in another CTA
    for k in (0, 256, 599):
        _set(f, o, *base)
        a, _, _, cr = _associate(f, o, _graze(o, k, n), n)
        assert a[0] == -1 and cr[0] == 0
    for kc in (256, 400, n):
        _set(f, o, *base)
        a, _, _, cr = _associate(f, o, FAR, kc)
        assert (a[0], cr[0]) == ((kc, 1) if kc < n else (-1, 0))
    for j in (41, 72, 296, 552):  # same warp, same lane of another warp, the next CTA, the CTA after
        _tie(f, o, 40, j, base)
    # a NaN landmark never wins, not even against a reading of where it was; the others associate as usual
    q = 300
    st = base[0].copy()
    st[3 + 2 * q] = np.nan
    _set(f, o, st, base[1])
    xy = np.stack([_robot_frame(base[0], q), _robot_frame(st, q + 1, (0.01, -0.005)), _robot_frame(st, 7)])
    a, _, _, _ = _associate(f, o, xy, n, nan_entry=3 + 2 * q)
    assert q not in a and a[1] == q + 1 and a[2] == 7


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_local_emulation(gpu_pkg, world):
    """n = 600 split over 2 or 3 emulated ranks (300 landmarks and two CTAs per rank, or 200 and one): each rank merges
    its CTAs, then the ranks' partials are merged.  Readings aim at the first and last landmark of every rank and at
    both sides of a rank's CTA boundary."""
    from ekf_slam_ml_b200.sharded import ShardedEKF
    n = 600
    f = ShardedEKF.local_emulation(n, world)
    o = _built(f, n)
    targets = []
    for g in range(world):
        r0, r1 = f.rows(g)
        first, last = (max(r0, 3) - 3) // 2, (r1 - 5) // 2
        targets += [first, last] + [k for k in (first + 255, first + 256) if k < last]
    assert len(set(targets)) == len(targets) == {2: 8, 3: 6}[world]  # 200 landmarks per rank at world = 3: one CTA
    for k in targets:
        a, _, _, cr = _associate(f, o, _robot_frame(o.state, k, (0.01, -0.005)), n)
        assert a[0] == k and cr[0] == 0
        a, _, _, cr = _associate(f, o, _graze(o, k, n), n)
        assert a[0] == -1 and cr[0] == 0
    a, _, _, cr = _associate(f, o, FAR, 256)
    assert a[0] == 256 and cr[0] == 1
    a, _, _, cr = _associate(f, o, -FAR, n)  # (not FAR: landmark 256 now sits there)
    assert a[0] == -1 and cr[0] == 0
