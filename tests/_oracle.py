"""ctypes bindings for the CPU checkers under oracle/ (test infrastructure only).

* ``RefEKF``     – the reference's own rigid2d::EKF_SLAM (oracle/_ref/libekf_ref.so, built from
                   the checkout EKF_SLAM_REFERENCE names by oracle/Makefile; present only where it was built).
* ``OracleEKF``  – the plain-C O(N^2) restatement (oracle/libekf_oracle.so, oracle/ekf_oracle.c).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import this module.
"""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
_dp = ctypes.POINTER(ctypes.c_double)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_i32p = ctypes.POINTER(ctypes.c_int32)


def _d(a):
    return a.ctypes.data_as(_dp)


def _u8(a):
    return a.ctypes.data_as(_u8p)


def build_oracle():
    """(Re)build oracle/libekf_oracle.so (and oracle/_ref when EKF_SLAM_REFERENCE names a reference checkout)."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "all"], check=True, stdout=subprocess.DEVNULL)


def _load(path):
    return ctypes.CDLL(path) if os.path.exists(path) else None


_oracle_lib = None
_ref_lib = None


def oracle_lib():
    global _oracle_lib
    if _oracle_lib is None:
        p = os.path.join(ORACLE_DIR, "libekf_oracle.so")
        if not os.path.exists(p):
            build_oracle()
        L = ctypes.CDLL(p)
        L.oracle_create.restype = ctypes.c_void_p
        L.oracle_maha.restype = ctypes.c_double
        L.oracle_normalize_angle.restype = ctypes.c_double
        L.oracle_normalize_angle.argtypes = [ctypes.c_double]
        L.oracle_run_known.restype = ctypes.c_int64
        _oracle_lib = L
    return _oracle_lib


def ref_lib():
    """The reference build, or None when oracle/_ref was never built here."""
    global _ref_lib
    if _ref_lib is None:
        L = _load(os.path.join(ORACLE_DIR, "_ref", "libekf_ref.so"))
        if L is None:
            return None
        L.ref_ekf_create.restype = ctypes.c_void_p
        L.ref_ekf_maha.restype = ctypes.c_double
        L.ref_normalize_angle.restype = ctypes.c_double
        L.ref_normalize_angle.argtypes = [ctypes.c_double]
        L.ref_bench_known.restype = ctypes.c_double
        L.ref_silence_stdout(1)
        L.ref_blas_threads(1)
        _ref_lib = L
    return _ref_lib


class OracleEKF:
    """Plain-C restatement; same verbs as rigid2d::EKF_SLAM."""

    def __init__(self, n):
        self.L = oracle_lib()
        self.n = int(n)
        self.N = 3 + 2 * self.n
        self.h = ctypes.c_void_p(self.L.oracle_create(self.n))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.oracle_destroy(self.h)
            self.h = None

    def prediction(self, dtheta, dx):
        self.L.oracle_prediction(self.h, ctypes.c_double(dtheta), ctypes.c_double(dx))

    def measurement(self, xy, visible):
        xy = np.ascontiguousarray(xy, dtype=np.float64)
        vis = np.ascontiguousarray(visible, dtype=np.uint8)
        assert xy.size == 2 * self.n and vis.size == self.n
        self.L.oracle_measurement(self.h, _d(xy), _u8(vis))

    def data_association(self, xy, known):
        """known: uint8[n], updated in place.  Returns (assoc, dmin, second, created)."""
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1)
        m = xy.size // 2
        assert known.dtype == np.uint8 and known.size == self.n
        assoc = np.full(m, -2, dtype=np.int32)
        dmin = np.zeros(m)
        second = np.zeros(m)
        created = np.zeros(m, dtype=np.uint8)
        self.L.oracle_data_association(self.h, _d(xy), ctypes.c_int(m), _u8(known),
                                       assoc.ctypes.data_as(_i32p), _d(dmin), _d(second), _u8(created))
        return assoc, dmin, second, created

    def maha(self, mx, my, i):
        return self.L.oracle_maha(self.h, ctypes.c_double(mx), ctypes.c_double(my), ctypes.c_int(i))

    @property
    def state(self):
        out = np.zeros(self.N)
        self.L.oracle_get_state(self.h, _d(out))
        return out

    @state.setter
    def state(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        self.L.oracle_set_state(self.h, _d(v))

    @property
    def sigma(self):
        out = np.zeros((self.N, self.N))
        self.L.oracle_get_sigma(self.h, _d(out))
        return out

    @sigma.setter
    def sigma(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        self.L.oracle_set_sigma(self.h, _d(v))

    @property
    def init_flag(self):
        return bool(self.L.oracle_get_init_flag(self.h))

    @init_flag.setter
    def init_flag(self, v):
        self.L.oracle_set_init_flag(self.h, ctypes.c_int(int(v)))


class RefEKF:
    """The reference's own class (dense N^3), through oracle/ref_driver.cpp."""

    def __init__(self, n):
        self.L = ref_lib()
        if self.L is None:
            raise RuntimeError("oracle/_ref/libekf_ref.so not built (set EKF_SLAM_REFERENCE to a reference checkout and build)")
        self.n = int(n)
        self.N = 3 + 2 * self.n
        self.h = ctypes.c_void_p(self.L.ref_ekf_create(self.n))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_ekf_destroy(self.h)
            self.h = None

    def prediction(self, dtheta, dx):
        self.L.ref_ekf_prediction(self.h, ctypes.c_double(dtheta), ctypes.c_double(dx))

    def measurement(self, xy, visible):
        xy = np.ascontiguousarray(xy, dtype=np.float64)
        vis = np.ascontiguousarray(visible, dtype=np.uint8)
        self.L.ref_ekf_measurement(self.h, _d(xy), _u8(vis))

    def data_association(self, xy, known):
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1)
        self.L.ref_ekf_data_association(self.h, _d(xy), ctypes.c_int(xy.size // 2), _u8(known))

    def maha(self, mx, my, i):
        return self.L.ref_ekf_maha(self.h, ctypes.c_double(mx), ctypes.c_double(my), ctypes.c_int(i))

    @property
    def state(self):
        out = np.zeros(self.N)
        self.L.ref_ekf_get_state(self.h, _d(out))
        return out

    @state.setter
    def state(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        self.L.ref_ekf_set_state(self.h, _d(v))

    @property
    def sigma(self):
        out = np.zeros((self.N, self.N))
        self.L.ref_ekf_get_sigma(self.h, _d(out))
        return out

    @sigma.setter
    def sigma(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        self.L.ref_ekf_set_sigma(self.h, _d(v))

    @property
    def init_flag(self):
        return bool(self.L.ref_ekf_get_init_flag(self.h))

    @init_flag.setter
    def init_flag(self, v):
        self.L.ref_ekf_set_init_flag(self.h, ctypes.c_int(int(v)))


def odometry_inputs():
    """The 4,000 seeded (pose, left, right) cases on which DiffDrive::updatePose is pinned (tests/golden/odometry.npz)."""
    rng = np.random.default_rng(5)
    for k in range(4000):
        pose = np.array([rng.normal(), rng.normal(), rng.uniform(-7, 7)])
        l, r = (rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2)) if k % 3 else (rng.uniform(-40, 40), rng.uniform(-40, 40))
        if k % 7 == 0:
            r = l + rng.uniform(-1e-6, 1e-6)  # below the 1e-4 rad "straight line" threshold
        yield pose, l, r


def sigma_err(a, b):
    """Scaled covariance error used everywhere in the parity tests (SURVEY.md §7 hard part 1):
    max_ab |a_ab - b_ab| / max(|b_ab|, sqrt(|b_aa b_bb|), tiny)."""
    d = np.sqrt(np.abs(np.diag(b)))
    scale = np.maximum(np.abs(b), np.outer(d, d))
    scale = np.maximum(scale, 1e-300)
    return float(np.max(np.abs(a - b) / scale))


def state_err(a, b):
    """max |a-b| / max(1, |b|)."""
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))))
