"""CPU suite (-m "not gpu"): host logic and the ABI surface — no compute calls (there is no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for h in ("ekf_slam_b200.h", "circle_fit_b200.h", "ekf_sharded_b200.h", "tube_world_b200.h"):
        p = os.path.join(ROOT, "include", h)
        if not os.path.exists(p):
            continue
        src = re.sub(r"/\*.*?\*/", "", open(p).read(), flags=re.S)
        names |= set(re.findall(r"\b((?:ekf|circles|tubeworld)_[a-z0-9_]+)\s*\(", src))
    return names


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg._lib.load()
    lib_sh = pkg._lib.load_sharded()
    decl = declared_symbols()
    assert len(decl) > 80
    missing = [n for n in sorted(decl) if not hasattr(lib_sh if n.startswith("ekf_sharded_") else lib, n)]
    assert not missing, missing
    # and the Python binding tables cover the same set (headers, libraries and bindings in step)
    bound = set(pkg._lib.SIGNATURES) | set(pkg._lib.SIGNATURES_SHARDED)
    assert bound == decl, bound ^ decl


NO_GPU = r'''
import sys
import numpy as np
import pytest
sys.path.insert(0, sys.argv[1])
import ekf_slam_ml_b200 as pkg
assert pkg.device_count() == 0
with pytest.raises(pkg.EkfError):
    pkg.EKF_SLAM(20)
with pytest.raises(pkg.EkfError):
    pkg.EKFBatch(8, 20)
with pytest.raises(pkg.EkfError):
    pkg.CircleFitting().run_batch(np.ones((1, 360), np.float32))
sys.stdout.write("no-gpu ok\n")
'''


def test_no_gpu_means_loud_failure_not_fallback():
    """In a process that sees no device (CUDA_VISIBLE_DEVICES empty, so this runs on a GPU machine too)."""
    r = subprocess.run([sys.executable, "-c", NO_GPU, ROOT], capture_output=True, text=True, timeout=240,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and "no-gpu ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_product_never_imports_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    pat = re.compile(r"oracle|_ref\b|libekf_ref|ekf_oracle")
    bad = []
    for d, _, files in os.walk(os.path.join(ROOT, "ekf-slam-ml_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")):
                txt = open(os.path.join(d, f), errors="ignore").read()
                for i, line in enumerate(txt.splitlines(), 1):
                    if pat.search(line) and "oracle" in line.lower() and "import" in line:
                        bad.append((f, i, line.strip()))
    for f in os.listdir(os.path.join(ROOT, "include")):
        p = os.path.join(ROOT, "include", f)
        if os.path.isfile(p) and "oracle/" in open(p).read():
            bad.append((f, 0, "mentions oracle/"))
    assert not bad, bad
    deps = subprocess.run(["ldd", os.path.join(ROOT, "ekf-slam-ml_b200", "libekfslam_b200.so")], capture_output=True,
                          text=True).stdout
    assert "oracle" not in deps and "openblas" not in deps


def test_body_twist_host_helper(pkg):
    g = np.load(os.path.join(ROOT, "tests", "golden", "helpers.npz"))
    for w, t in zip(g["wheels"], g["twists"]):
        tw = pkg.body_twist(0.16, 0.033, w[0], w[1])
        assert tw.angular() == t[0] and tw.linearX() == t[1] and tw.linearY() == 0.0


def test_tracegen_is_deterministic_and_batch_independent(pkg):
    tg = pkg.tracegen
    w = tg.dense_world(20)
    assert w.n_tubes == 20
    a = tg.simulate_known(w, 6, 8, seed=9)
    b = tg.simulate_known(w, 2, 8, seed=9, first_filter=3)
    c = tg.simulate_known(w, 64, 8, seed=9, workers=4)
    for k in a:
        assert np.array_equal(a[k][:, 3:5], b[k])
        assert np.array_equal(a[k], c[k][:, :6])
    assert a["vis"][0].sum() == 0 and a["vis"][1:].sum() > 0          # first node cycle only initialises
    d = np.hypot(a["truth"][..., 0], a["truth"][..., 1] - 0.2)        # follow_circle: R = 0.2 about (0, 0.2)
    assert np.all(np.abs(d - 0.2) < 0.05)
    u = tg.simulate_unknown(w, 3, 5, seed=1, m_max=6)
    assert u["meas"].shape == (5, 3, 6, 2) and u["count"].max() <= 6
    s = tg.simulate_scans(tg.default_world(), 2, 5, seed=2)
    assert s["ranges"].dtype == np.float32 and s["ranges"].shape == (5, 2, 360)
    assert np.all(s["ranges"] < 3.6) and list(s["scan_id"]) == [0, 0, 1, 1, 2]


def test_row_block_partition(pkg):
    sh = pkg.sharding
    for N, G, al in ((80003, 8, 16), (16387, 2, 16), (43, 4, 1), (203, 8, 16)):
        b = sh.row_blocks(N, G, al)
        assert b[0] == 0 and b[-1] == N and all(x <= y for x, y in zip(b, b[1:]))
        assert all(x % al == 0 or x == N for x in b)
        for row in (0, 1, 2, N // 2, N - 1):
            g = sh.owner_of_row(row, b)
            assert b[g] <= row < b[g + 1]


def test_landmark_row_partition_matches_engine_contract(pkg):
    sh = pkg.sharding
    for n, G in ((40000, 8), (40000, 2), (20, 3), (61, 4), (8192, 8)):
        b = sh.landmark_row_blocks(n, G)
        N = 3 + 2 * n
        assert b[0] == 0 and b[-1] == N and len(b) == G + 1
        assert all(x < y for x, y in zip(b, b[1:]))
        assert all(x % 2 == 1 for x in b[1:])          # landmark row pairs (3+2i, 4+2i) are never split
        assert sh.owner_of_row(0, b) == 0 and sh.owner_of_row(2, b) == 0
        for i in (0, n // 2, n - 1):
            assert sh.owner_of_row(3 + 2 * i, b) == sh.owner_of_row(4 + 2 * i, b)


WORKER = r'''
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
import ekf_slam_ml_b200 as pkg
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
tg, sh = pkg.tracegen, pkg.sharding
first, per = sh.filter_range(rank, world, 5)
tr = tg.simulate_known(tg.default_world(20), per, 6, seed=4, first_filter=first)
whole = tg.simulate_known(tg.default_world(20), per * world, 6, seed=4)
assert np.array_equal(tr["xy"], whole["xy"][:, first:first + per])          # shards tile the global batch
# per-rank error statistic -> all-reduce == statistic of the whole batch
est = tr["truth"][-1] + 0.01 * (rank + 1)
d = est - tr["truth"][-1]
local = np.array([np.sum(d[:, 0] ** 2), np.sum(d[:, 1] ** 2), np.sum(d[:, 2] ** 2), per], dtype=np.float64)
tot = sh.allreduce_sum(local, dist)
exp = np.array([sum(per * (0.01 * (r + 1)) ** 2 for r in range(world))] * 3 + [per * world])
assert np.allclose(tot, exp), (tot, exp)
assert sh.allreduce_max(float(rank + 1), dist) == float(world)
b = sh.row_blocks(203, world, 16)
rows = np.arange(b[rank], b[rank + 1])
cnt = sh.allreduce_sum(np.array([rows.size], dtype=np.float64), dist)
assert int(cnt[0]) == 203
dist.barrier()
dist.destroy_process_group()
sys.stdout.write("rank %d ok\n" % rank)  # one write: two ranks share the pipe
sys.stdout.flush()
'''


def test_two_rank_sharding_over_gloo(tmp_path):
    """World size 2 on CPU (gloo): filter sharding tiles the global batch, statistics all-reduce, max-over-ranks."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    import socket
    with socket.socket() as sk:  # a free rendezvous port (a fixed one can still sit in TIME_WAIT from an earlier run)
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script), ROOT],
                       capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "rank 0 ok" in r.stdout and "rank 1 ok" in r.stdout


def test_marker_list_is_the_visible_subset_in_id_order(pkg):
    """Host helper of ekf_batch_step_known_sparse: dense fake-sensor arrays -> CSR marker list."""
    rng = np.random.default_rng(3)
    B, n = 37, 23
    xy = rng.normal(size=(B, 2 * n))
    vis = (rng.random((B, n)) < 0.3).astype(np.uint8)
    vis[5] = 0                                   # a robot that sees nothing
    off, ids, pts = pkg.marker_list(xy, vis)
    assert off.dtype == np.int32 and ids.dtype == np.uint8 and pts.dtype == np.float64 and pts.flags.c_contiguous
    assert off[0] == 0 and off[-1] == vis.sum() == len(ids) == len(pts) and off[5] == off[6]
    for b in range(B):
        want = np.nonzero(vis[b])[0]
        assert np.array_equal(ids[off[b]:off[b + 1]], want)
        assert np.array_equal(pts[off[b]:off[b + 1]], xy[b].reshape(n, 2)[want])
    with pytest.raises(ValueError):
        pkg.marker_list(np.zeros((1, 600)), np.ones((1, 300), np.uint8))


def test_accuracy_report_formatting(pkg):
    r = {"robots": 2, "steps": 3, "seed": 0, "updates": 11, "landmark_rmse": 0.01, "landmarks": 20,
         "rmse_xytheta": {"slam": [0.001, 0.002, 0.01], "prediction_only": [0.1, 0.2, 0.3], "wheel_odometry": [0, 0, 0]},
         "worst_xy_error": {"slam": 0.004, "prediction_only": 0.3, "wheel_odometry": 0.0}}
    md = pkg.report.markdown(r)
    assert md.count("\n") >= 6 and "Slam | 0.00100 | 0.00200" in md and "Prediction only" in md
