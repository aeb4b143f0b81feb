"""The multi-factor covariance sweep (csrc/ekf_large_mma.cuh) at every depth P = 1..20 and at the edges of its geometry,
in the streamed single filter and in every rank of the row-sharded filter.

The traces here control how many corrections each call makes: call 0 lists every slot, then every count c = 1..20
(at most n) comes once per round, two rounds in two seeded orders.  With max_pending = 20 and the pending factors cut
at the end of each call, call t ends in exactly one sweep with P = c_t, which the tests assert through sweep_count.
Each run is held bit for bit to the same filter at max_pending = 1 (one sweep per correction on the register path) and
to the CPU oracle at 1e-9."""
import functools
import os
import re

import numpy as np
import pytest

import _single as single
from _batch import sms
from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9
MAX_P = 20  # the deepest group (kMaxPending)

# SweepTile<P>: (tile columns, stage rows) up to P = 14 and from P = 15 on; 128-row work units; eight consumer warps
# share a tile's columns.  Checked against the header below, so that a change of the geometry fails here loudly.
NARROW_MAX_P = 14
TILES = ((512, 8), (256, 16))
UNIT_ROWS = 128
CONSUMER_WARPS = 8


def _header_geometry():
    with open(os.path.join(ROOT, "ekf-slam-ml_b200", "csrc", "ekf_large_mma.cuh")) as fh:
        src = fh.read()
    cols = re.search(r"COLS = P <= (\d+) \? (\d+) : (\d+);", src)
    srows = re.search(r"SROWS = P <= (\d+) \? (\d+) : (\d+);", src)
    unit = re.search(r"kUnitRows = (\d+);", src)
    warps = re.search(r"kTmaConsumerWarps = (\d+);", src)
    assert cols and srows and unit and warps, "SweepTile<P> is no longer written as this test reads it"
    assert cols.group(1) == srows.group(1)
    return (int(cols.group(1)), ((int(cols.group(2)), int(srows.group(2))), (int(cols.group(3)), int(srows.group(3)))),
            int(unit.group(1)), int(warps.group(1)))


def _geometry(n):
    """What a sweep over the streamed filter's Sigma meets at map size n, per tile geometry (COLS, SROWS): the width of
    the last tile, the consumer warps that have blocks in it, the rows of the last stage and the work units."""
    N = 3 + 2 * n
    ld = -(-N // 16) * 16
    units = -(-N // UNIT_ROWS)
    last_unit = N - UNIT_ROWS * (units - 1)
    tail, warps, stage, work = [], [], [], []
    for cols, srows in TILES:
        w = ld % cols or cols
        tail.append(w)
        warps.append(-(-w // (cols // CONSUMER_WARPS)))
        stage.append(last_unit % srows or srows)
        work.append(-(-ld // cols) * units)
    return N, ld, tuple(tail), tuple(warps), last_unit, tuple(stage), tuple(work)


# Per geometry, (P <= 14, P >= 15):  last tile's width, consumer warps with blocks in it, rows of the last stage, units.
SHAPES = [
    # n,    N,    ld,    last tile   warps    last unit  last stage  work units   what it reaches
    (1,     5,    16,   (16, 16),   (1, 1),    5,       (5, 5),     (1, 1)),     # one 16-wide tile, a 5-row stage
    (6,     15,   16,   (16, 16),   (1, 1),    15,      (7, 15),    (1, 1)),     # one pad column
    (62,    127,  128,  (128, 128), (2, 4),    127,     (7, 15),    (1, 1)),     # one unit, one row short of full
    (63,    129,  144,  (144, 144), (3, 5),    1,       (1, 1),     (2, 2)),     # a second unit of one row
    (126,   255,  256,  (256, 256), (4, 8),    127,     (7, 15),    (2, 2)),     # exactly one 256-column tile
    (127,   257,  272,  (272, 16),  (5, 1),    1,       (1, 1),     (3, 6)),     # 16-wide tail: warp 0 alone at P >= 15
    (254,   511,  512,  (512, 256), (8, 8),    127,     (7, 15),    (4, 8)),     # exactly one / two full tiles
    (255,   513,  528,  (16, 16),   (1, 1),    1,       (1, 1),     (10, 15)),   # 16-wide tail at both widths
    (502,   1007, 1008, (496, 240), (8, 8),    111,     (7, 15),    (16, 32)),   # wide tails, last warp partial
    (2500,  5003, 5008, (400, 144), (7, 5),    11,      (3, 11),    (400, 800)),  # every CTA runs >= 2 units
]
MULTI_UNIT_N = SHAPES[-1][0]
assert _header_geometry() == (NARROW_MAX_P, TILES, UNIT_ROWS, CONSUMER_WARPS), "the sweep's geometry changed: revisit SHAPES"
for _row in SHAPES:
    assert _geometry(_row[0]) == tuple(_row[1:]), _row

# Row-sharded filter: (n, world) -> the rows of each rank (csrc/sharded/sharded.cu::partition)
SHARDED = {
    (20, 8): (9, 6, 6, 6, 6, 6, 4, 0),          # one empty rank
    (9, 8): (7, 4, 4, 4, 2, 0, 0, 0),           # three empty ranks and a one-landmark rank
    (13, 6): (9, 6, 6, 6, 2, 0),                # empty last rank
    (61, 4): (35, 32, 32, 26),                  # every rank but the first starts at an odd row
    (400, 8): (103,) + (100,) * 7,              # 100-row ranks starting at odd rows
}
SHARDED_DEPTHS = (1, 2, 3, 14, 15, 20)


def _world(pkg, n):
    """n landmarks on a near-square grid (the last row partly filled)."""
    nx = int(np.ceil(np.sqrt(n)))
    w = pkg.tracegen.grid_world(nx, -(-n // nx), pitch=0.35, n_slots=n)
    w.tubes_x, w.tubes_y = w.tubes_x[:n], w.tubes_y[:n]
    return w


def controlled_trace(pkg, n, seed):
    """A simulated known-association trace whose call t has exactly c_t visible slots.  Call 0 lists every slot (each
    landmark starts at its reading and is corrected once); then rounds of the counts 1..min(20, n), each round in its
    own seeded order: two rounds, and more while the corrections could not fill three groups of 20 (small maps).  The
    simulator's fake sensor reads every tube, so any set of slots has consistent readings; every fourth set contains
    slot 0, slot n - 1, both, or neither on purpose (the first and the last, partial stage of a sweep)."""
    C = min(MAX_P, n)
    rng = np.random.default_rng(seed)
    counts = []
    while len(counts) < 2 * C or sum(counts) < 3 * MAX_P:
        counts += [int(c) for c in rng.permutation(np.arange(1, C + 1))]
    T = 1 + len(counts)
    tr = pkg.tracegen.simulate_known(_world(pkg, n), 1, T, seed=seed)
    vis = np.zeros((T, 1, n), np.uint8)
    vis[0] = 1
    for t, c in enumerate(counts, 1):
        ends = np.array(list(dict.fromkeys(((), (0,), (n - 1,), (0, n - 1))[t % 4]))[:c], dtype=np.int64)
        rest = rng.choice(np.setdiff1d(np.arange(n), ends), c - len(ends), replace=False)
        vis[t, 0, ends] = 1
        vis[t, 0, rest] = 1
    assert np.array_equal(vis[1:, 0].sum(axis=1), counts)
    if n > 1:
        first, last = vis[1:, 0, 0] == 1, vis[1:, 0, n - 1] == 1
        assert (first & ~last).any() and (last & ~first).any() and (first & last).any()
    return {"twists": tr["twists"], "xy": tr["xy"], "vis": vis}


@functools.lru_cache(maxsize=None)
def _trace(pkg, n):
    return controlled_trace(pkg, n, seed=n)


@functools.lru_cache(maxsize=None)
def _oracle_end(pkg, n):
    """The oracle's state and Sigma after the whole controlled trace of n (one run per session: at n = 2,500 it is
    the slowest part of this file)."""
    o = single.run_known(OracleEKF(n), _trace(pkg, n))
    return o.state, o.sigma


def _streamed(pkg, n, max_pending, carry):
    f = pkg.EKF_SLAM(n, engine=pkg.ENGINE_STREAM)
    f.set_max_pending(max_pending)
    f.set_carry_pending(carry)
    return f


def _same_bits(a, b, what):
    assert np.array_equal(single.bits(a), single.bits(b)), what


@pytest.mark.parametrize("n", [row[0] for row in SHAPES])
def test_streamed_sweep_at_every_depth_is_bit_identical(gpu_pkg, n):
    """Filter a (max_pending 20) sweeps once per call with P = the call's count; filter b (max_pending 1) sweeps once
    per correction.  Bit-identical after every call (every fourth at n = 2,500, where Sigma is 200 MB), and filter a
    within 1e-9 of the oracle at the end."""
    if n == MULTI_UNIT_N:
        assert min(_geometry(n)[-1]) >= 2 * sms(), "raise n: some CTA of the sweep runs a single work unit"
    tr = _trace(gpu_pkg, n)
    T = tr["vis"].shape[0]
    every = 4 if n == MULTI_UNIT_N else 1
    a, b = _streamed(gpu_pkg, n, MAX_P, False), _streamed(gpu_pkg, n, 1, False)
    for t in range(T):
        sa, sb = a.sweep_count, b.sweep_count
        single.step_known(a, tr, t)
        single.step_known(b, tr, t)
        c = int(tr["vis"][t, 0].sum())
        assert a.sweep_count - sa == (1 if t else -(-n // MAX_P)), t  # call t > 0: one sweep, P = c
        assert b.sweep_count - sb == c, t
        if t % every == 0 or t == T - 1:
            _same_bits(a.state, b.state, ("state", t))
            _same_bits(a.sigma, b.sigma, ("sigma", t))
    assert a.update_count == b.update_count == int(tr["vis"].sum())
    x, s = _oracle_end(gpu_pkg, n)
    ex, es = state_err(a.state, x), sigma_err(a.sigma, s)
    assert ex < TOL and es < TOL, (ex, es)


@pytest.mark.parametrize("n", [1, 6, MULTI_UNIT_N])
def test_streamed_sweep_with_groups_carried_across_calls(gpu_pkg, n):
    """The default schedule: groups run to max_pending corrections across calls and predictions, and the getters settle
    the last one.  At n = 1 and 6 this is what reaches the DMMA sweep and its 256-column geometry.  Same filter as the
    per-call schedule to rounding (bounds of test_pending_factors_carried_across_prediction), and as the oracle."""
    tr = _trace(gpu_pkg, n)
    total = int(tr["vis"].sum())
    ref = single.run_known(_streamed(gpu_pkg, n, MAX_P, False), tr)
    xr, sr = ref.state, ref.sigma
    ref.close()
    xo, so = _oracle_end(gpu_pkg, n)
    for k in (3, 14, 15, 20):
        f = single.run_known(_streamed(gpu_pkg, n, k, True), tr)
        assert f.sweep_count == total // k, k  # every sweep so far had exactly k factors
        x, s = f.state, f.sigma
        assert f.sweep_count == -(-total // k) and f.update_count == total, k
        assert state_err(x, xr) < 1e-12 and sigma_err(s, sr) < 1e-11, k
        ex, es = state_err(x, xo), sigma_err(s, so)
        assert ex < TOL and es < TOL, (k, ex, es)
        f.close()


@pytest.mark.parametrize("n,world", list(SHARDED))
def test_sharded_sweep_at_every_depth_and_with_empty_ranks(gpu_pkg, n, world):
    """Local emulation of the row-sharded filter at max_pending 1, 2, 3, 14, 15 and 20, per-call groups: each rank
    sweeps its own rows from row0 = its first row (ranks without rows skip the sweep).  Every depth is bit-identical to
    depth 1 after every call and within 1e-9 of the oracle."""
    from ekf_slam_ml_b200.sharded import ShardedEKF
    N = 3 + 2 * n
    tr = _trace(gpu_pkg, n)
    fs = []
    for k in SHARDED_DEPTHS:
        f = ShardedEKF.local_emulation(n, world)
        f.set_max_pending(k)
        f.set_carry_pending(False)
        fs.append(f)
    bounds = gpu_pkg.sharding.landmark_row_blocks(n, world)
    assert [fs[0].rows(g) for g in range(world)] == list(zip(bounds[:-1], bounds[1:]))
    assert tuple(np.diff(bounds)) == SHARDED[n, world] and bounds[-1] == N  # an empty rank owns (N, N)
    for t in range(tr["vis"].shape[0]):
        c = int(tr["vis"][t, 0].sum())
        for f, k in zip(fs, SHARDED_DEPTHS):
            s0 = f.sweep_count
            single.step_known(f, tr, t)
            assert f.sweep_count - s0 == -(-c // k), (k, t)
        x1, s1 = fs[0].state, fs[0].sigma_full_local()
        for f, k in zip(fs[1:], SHARDED_DEPTHS[1:]):
            _same_bits(f.state, x1, ("state", k, t))
            _same_bits(f.sigma_full_local(), s1, ("sigma", k, t))
    xo, so = _oracle_end(gpu_pkg, n)
    for f, k in zip(fs, SHARDED_DEPTHS):
        assert f.update_count == int(tr["vis"].sum()), k
        ex, es = state_err(f.state, xo), sigma_err(f.sigma_full_local(), so)
        assert ex < TOL and es < TOL, (k, ex, es)
        f.close()
