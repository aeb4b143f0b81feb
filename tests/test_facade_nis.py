"""The NIS read-out of the C++ facade (rigid2d::EKF_SLAM::set_nis / nis / last_nis, include/rigid2d/ekf_slam.hpp):
tests/cpp/facade_nis_test.cpp drives it as a SLAM node would, copy-assignment included."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    """Compiles the facade test into tmp_path: the checkout may be read-only for the user running the tests."""
    exe = str(tmp_path / "facade_nis_test")
    cmd = ["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "facade_nis_test.cpp"), "-o", exe,
           "-L" + os.path.join(ROOT, "ekf-slam-ml_b200"), "-lekfslam_b200",
           "-Wl,-rpath," + os.path.join(ROOT, "ekf-slam-ml_b200")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_facade_nis_compiles_against_the_c_abi(pkg, tmp_path):
    pkg._lib.load()
    exe = _build(tmp_path)
    assert os.path.exists(exe)
    if pkg.device_count() == 0:  # no GPU here: the facade must report the failure, not pretend to work
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode != 0 and "ekf_create failed" in r.stderr


@pytest.mark.gpu
def test_facade_nis_runs(gpu_pkg, tmp_path):
    exe = _build(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "FACADE NIS OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
