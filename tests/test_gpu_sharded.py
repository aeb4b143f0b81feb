"""Row-block-sharded covariance (cfg5 engine).  On one GPU the `world` ranks are emulated inside one process
(exchanges become device copies) so that the partition / partial-W / gathered-K / merged-argmin arithmetic is checked
against the oracle; with >= 2 GPUs the same trace runs through real NCCL ranks (torchrun) and must give the same state."""
import os
import subprocess
import sys

import numpy as np
import pytest

from _oracle import OracleEKF, sigma_err, state_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9


def _world(pkg, n):
    tg = pkg.tracegen
    nx = int(np.ceil(np.sqrt(n)))
    ny = -(-n // nx)
    w = tg.grid_world(nx, ny, pitch=0.45, n_slots=n, max_visible=1.0)
    w.tubes_x, w.tubes_y = w.tubes_x[:n], w.tubes_y[:n]
    return w


@pytest.mark.parametrize("n,world", [(20, 1), (20, 3), (61, 4), (400, 2), (400, 8)])
def test_local_emulation_known_association(gpu_pkg, n, world):
    from ekf_slam_ml_b200.sharded import ShardedEKF
    tg = gpu_pkg.tracegen
    tr = tg.simulate_known(_world(gpu_pkg, n), 1, 10, seed=n + world)
    f = ShardedEKF.local_emulation(n, world)
    o = OracleEKF(n)
    # partition: landmark row pairs are never split, rank 0 owns the robot rows, blocks tile [0, N)
    bounds = [f.rows(g) for g in range(world)]
    assert bounds[0][0] == 0 and bounds[-1][1] == f.N
    assert all(bounds[g][1] == bounds[g + 1][0] for g in range(world - 1))
    assert all(b[0] % 2 == 1 for b in bounds[1:])
    assert [b[0] for b in bounds] + [f.N] == gpu_pkg.sharding.landmark_row_blocks(n, world)
    worst = 0.0
    for t in range(10):
        f.prediction(tuple(tr["twists"][t, 0]))
        o.prediction(*tr["twists"][t, 0])
        f.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        o.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
        if t % 3 == 0 or t == 9:
            worst = max(worst, state_err(f.state, o.state), sigma_err(f.sigma_full_local(), o.sigma))
    assert f.update_count == int(tr["vis"].sum()) > 10
    assert worst < TOL, worst


@pytest.mark.parametrize("n,world", [(20, 2), (20, 4), (150, 3)])
def test_local_emulation_unknown_association(gpu_pkg, n, world):
    from ekf_slam_ml_b200.sharded import ShardedEKF
    tg = gpu_pkg.tracegen
    w = _world(gpu_pkg, n) if n > 20 else tg.default_world(20)
    tr = tg.simulate_unknown(w, 1, 25, seed=7 + n, m_max=12)
    f = ShardedEKF.local_emulation(n, world)
    o = OracleEKF(n)
    kf, ko = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for t in range(25):
        f.prediction(tuple(tr["twists"][t, 0]))
        o.prediction(*tr["twists"][t, 0])
        m = int(tr["count"][t, 0])
        if m == 0:
            continue
        r = f.data_association(tr["meas"][t, 0, :m], kf)
        a, dmin, sec, cr = o.data_association(tr["meas"][t, 0, :m], ko)
        assert np.array_equal(r["assoc"], a) and np.array_equal(r["created"], cr) and np.array_equal(kf, ko)
        np.testing.assert_allclose(r["dmin"], dmin, rtol=1e-7, atol=1e-9)
    assert ko.sum() >= 4
    assert state_err(f.state, o.state) < TOL and sigma_err(f.sigma_full_local(), o.sigma) < TOL


NCCL_WORKER = r'''
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import torch, torch.distributed as dist
import ekf_slam_ml_b200 as pkg
from ekf_slam_ml_b200.sharded import ShardedEKF
from _oracle import OracleEKF, sigma_err, state_err
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, world = dist.get_rank(), dist.get_world_size()
n = 300
tg = pkg.tracegen
nx = 20
w = tg.grid_world(nx, 15, pitch=0.45, n_slots=n, max_visible=1.0)
tr = tg.simulate_known(w, 1, 8, seed=5)
tu = tg.simulate_unknown(w, 1, 3, seed=6, m_max=8)
f = ShardedEKF.from_process_group(n, dist, local)
o = OracleEKF(n)
for t in range(8):
    f.prediction(tuple(tr["twists"][t, 0])); o.prediction(*tr["twists"][t, 0])
    f.measurement(tr["xy"][t, 0], tr["vis"][t, 0]); o.measurement(tr["xy"][t, 0], tr["vis"][t, 0])
kf, ko = np.ones(n, np.uint8), np.ones(n, np.uint8)
for t in range(3):
    m = int(tu["count"][t, 0])
    r = f.data_association(tu["meas"][t, 0, :m], kf)
    a, dmin, sec, cr = o.data_association(tu["meas"][t, 0, :m], ko)
    assert np.array_equal(r["assoc"], a), (r["assoc"], a)
a, b = f.rows(0)
err_s = sigma_err_rows = float(np.max(np.abs(f.sigma_rows(0) - o.sigma[a:b]) / np.maximum(np.maximum(np.abs(o.sigma[a:b]), np.sqrt(np.abs(np.outer(np.diag(o.sigma)[a:b], np.diag(o.sigma))))), 1e-300)))
err_x = state_err(f.state, o.state)
assert err_x < 1e-9 and err_s < 1e-9, (rank, err_x, err_s)
dist.barrier()
sys.stdout.write("RANK%dOK rows=(%d,%d) err_state=%.2e err_sigma=%.2e exchange=%s\n" % (rank, a, b, err_x, err_s, f.exchange)); sys.stdout.flush()
f.close()
dist.destroy_process_group()
'''


# EKF_SHARDED_EXCHANGE selects the W exchange: unset = the push over NVLink (multicast where the fabric has it),
# push-unicast = the push by peer stores, nccl = the NCCL all-reduce.
@pytest.mark.parametrize("mode,expected,port", [
    (None, "exchange=push over NVLink (", 29688),
    ("push-unicast", "exchange=push over NVLink (peer stores)", 29689),
    ("nccl", "exchange=nccl all-reduce", 29690),
], ids=["default", "push-unicast", "nccl"])
def test_nccl_two_ranks(gpu_pkg, tmp_path, mode, expected, port):
    """Real NCCL ranks, one per GPU (needs >= 2 GPUs), in each exchange mode."""
    if gpu_pkg.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(NCCL_WORKER)
    env = {k: v for k, v in os.environ.items() if k != "EKF_SHARDED_EXCHANGE"}
    if mode:
        env["EKF_SHARDED_EXCHANGE"] = mode
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script), ROOT],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "RANK0OK" in r.stdout and "RANK1OK" in r.stdout, r.stdout[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RANK")]
    assert len(lines) == 2 and all(expected in ln for ln in lines), (expected, lines)
