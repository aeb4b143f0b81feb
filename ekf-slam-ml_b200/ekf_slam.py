"""Python mirror of the reference's rigid2d::EKF_SLAM call surface (rigid2d/include/rigid2d/ekf_slam.hpp:19-91)
over the C ABI — same method names, argument meaning and (absence of) error behaviour, so that parity
tests read like tests of the reference class.  All arithmetic happens in the CUDA library."""
import ctypes

import numpy as np

from . import _lib
from ._lib import c_double_p, c_i32_p, c_u8_p, check

ENGINE_AUTO, ENGINE_FUSED, ENGINE_STREAM = 0, 1, 2


class Vector2D:
    """rigid2d::Vector2D (rigid2d.hpp:68-107): plain {x, y} carrier."""
    __slots__ = ("x", "y")

    def __init__(self, x=0.0, y=0.0):
        self.x = float(x)
        self.y = float(y)


class Twist2D:
    """rigid2d::Twist2D (rigid2d.hpp:162-190, rigid2d.cpp:100-131)."""

    def __init__(self, angular=0.0, linear=None):
        self._ang = float(angular)
        self._lin = linear if linear is not None else Vector2D()

    def angular(self):
        return self._ang

    def linearX(self):
        return self._lin.x

    def linearY(self):
        return self._lin.y


def body_twist(wheel_base, wheel_radius, left, right):
    """DiffDrive::getBodyTwistForUpdate (diff_drive.cpp:38-47) -> Twist2D."""
    out = np.zeros(2)
    check(_lib.load().ekf_body_twist(wheel_base, wheel_radius, left, right, out.ctypes.data_as(c_double_p)))
    return Twist2D(out[0], Vector2D(out[1], 0.0))


def update_pose(wheel_base, wheel_radius, poses, left, right):
    """DiffDrive::updatePose (diff_drive.cpp:50-67) for a batch of odometers, evaluated by the device twin:
    poses [count, 3] = {x, y, theta}, wheel angle increments left / right [count] -> new poses."""
    p = np.array(poses, dtype=np.float64).reshape(-1, 3)
    l = np.ascontiguousarray(left, dtype=np.float64).reshape(-1)
    r = np.ascontiguousarray(right, dtype=np.float64).reshape(-1)
    assert l.size == r.size == p.shape[0]
    check(_lib.load().ekf_update_pose(float(wheel_base), float(wheel_radius), p.shape[0], p.ctypes.data, l.ctypes.data,
                                      r.ctypes.data))
    return p


class DiffDrive:
    """Mirror of rigid2d::DiffDrive's odometry side (diff_drive.hpp:18-60): dead-reckoning pose from wheel angles."""

    def __init__(self, wheel_base, wheel_radius, init_pos=(0.0, 0.0), init_theta=0.0):
        self.wheel_b, self.wheel_r = float(wheel_base), float(wheel_radius)
        self._pose = np.array([[init_pos[0], init_pos[1], init_theta]], dtype=np.float64)

    def getBodyTwistForUpdate(self, left_angle, right_angle):
        return body_twist(self.wheel_b, self.wheel_r, left_angle, right_angle)

    def updatePose(self, left_angle, right_angle):
        self._pose = update_pose(self.wheel_b, self.wheel_r, self._pose, [left_angle], [right_angle])

    def getPosition(self):
        return Vector2D(self._pose[0, 0], self._pose[0, 1])

    def getTheta(self):
        return float(self._pose[0, 2])


def normalize_angle(values, device=0):
    """rigid2d::normalize_angle (rigid2d.cpp:336-345) evaluated by the device twin."""
    a = np.ascontiguousarray(values, dtype=np.float64).reshape(-1)
    out = np.empty_like(a)
    check(_lib.load().ekf_normalize_angles(a.ctypes.data_as(c_double_p), out.ctypes.data_as(c_double_p), a.size, device))
    return out.reshape(np.shape(values))


def _as_xy(measures):
    if len(measures) and isinstance(measures[0], Vector2D):
        return np.array([[v.x, v.y] for v in measures], dtype=np.float64).reshape(-1)
    return np.ascontiguousarray(measures, dtype=np.float64).reshape(-1)


class EKF_SLAM:
    """Drop-in for rigid2d::EKF_SLAM.  `engine` picks the fused on-chip kernel or the HBM-streamed path."""

    def __init__(self, n_measurements, device=0, engine=ENGINE_AUTO):
        self._L = _lib.load()
        self.n = int(n_measurements)
        self.N = 3 + 2 * self.n
        h = ctypes.c_void_p()
        check(self._L.ekf_create_ex(self.n, device, engine, ctypes.byref(h)))
        self._h = h
        self.last_assoc = None
        self._pose_cache = None

    def close(self):
        if getattr(self, "_h", None):
            self._L.ekf_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def engine(self):
        return self._L.ekf_engine(self._h)

    # --- the reference's public surface
    def prediction(self, twist):
        """ekf_slam.cpp:55-106; accepts a Twist2D or a (dtheta, dx) pair."""
        if isinstance(twist, Twist2D):
            dth, dx = twist.angular(), twist.linearX()
        else:
            dth, dx = twist
        self._pose_cache = None
        check(self._L.ekf_predict(self._h, float(dth), float(dx)))

    def measurement(self, sensor_reading, visible_list, known_list=None):
        """ekf_slam.cpp:108-197.  known_list is accepted and ignored, exactly like the reference."""
        xy = np.ascontiguousarray(sensor_reading, dtype=np.float64).reshape(-1)
        vis = np.ascontiguousarray(visible_list, dtype=np.uint8).reshape(-1)
        if xy.size != 2 * self.n or vis.size != self.n:
            raise ValueError("sensor_reading must hold 2n values and visible_list n flags")
        self._pose_cache = None
        check(self._L.ekf_measurement(self._h, xy.ctypes.data_as(c_double_p), vis.ctypes.data_as(c_u8_p)))

    def data_association(self, measures, known_list):
        """ekf_slam.cpp:278-402.  known_list (uint8 ndarray or list) is updated in place like the reference's
        vector<bool>&.  Returns a dict with the per-measurement association log."""
        xy = _as_xy(measures)
        m = xy.size // 2
        known = np.ascontiguousarray(known_list, dtype=np.uint8).reshape(-1).copy()
        if known.size != self.n:
            raise ValueError("known_list must hold n flags")
        assoc = np.full(m, -2, dtype=np.int32)
        dmin = np.zeros(m)
        second = np.zeros(m)
        created = np.zeros(m, dtype=np.uint8)
        self._pose_cache = None
        check(self._L.ekf_data_association(self._h, xy.ctypes.data_as(c_double_p), m, known.ctypes.data_as(c_u8_p),
                                           assoc.ctypes.data_as(c_i32_p), dmin.ctypes.data_as(c_double_p),
                                           second.ctypes.data_as(c_double_p), created.ctypes.data_as(c_u8_p)))
        if isinstance(known_list, np.ndarray):
            known_list[...] = known.astype(known_list.dtype).reshape(known_list.shape)
        else:
            for i in range(self.n):
                known_list[i] = bool(known[i])
        self.last_assoc = {"assoc": assoc, "dmin": dmin, "second": second, "created": created}
        return self.last_assoc

    def getStateX(self):
        return float(self._pose()[1])

    def getStateY(self):
        return float(self._pose()[2])

    def getStateTheta(self):
        return float(self._pose()[0])

    def getStateLandmark(self):
        out = np.zeros(2 * self.n)
        check(self._L.ekf_get_landmarks(self._h, out.ctypes.data_as(c_double_p)))
        return out.reshape(-1, 1)

    # --- seams for parity tests / checkpointing (no reference counterpart; state and sigma are private there)
    def _pose(self):
        # x, y and theta are read one after the other (slam.cpp:433-434): one device read serves all three
        if self._pose_cache is None:
            out = np.zeros(3)
            check(self._L.ekf_get_pose(self._h, out.ctypes.data_as(c_double_p)))
            self._pose_cache = out
        return self._pose_cache

    def calculate_maha_dis(self, measure, ith_tube):
        mx, my = (measure.x, measure.y) if isinstance(measure, Vector2D) else measure
        d = ctypes.c_double()
        check(self._L.ekf_maha(self._h, float(mx), float(my), int(ith_tube), ctypes.byref(d)))
        return d.value

    @property
    def state(self):
        out = np.zeros(self.N)
        check(self._L.ekf_get_state(self._h, out.ctypes.data_as(c_double_p)))
        return out

    @state.setter
    def state(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(-1)
        assert v.size == self.N
        self._pose_cache = None
        check(self._L.ekf_set_state(self._h, v.ctypes.data_as(c_double_p)))

    @property
    def sigma(self):
        out = np.zeros((self.N, self.N))
        check(self._L.ekf_get_sigma(self._h, out.ctypes.data_as(c_double_p), self.N))
        return out

    @sigma.setter
    def sigma(self, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        assert v.shape == (self.N, self.N)
        check(self._L.ekf_set_sigma(self._h, v.ctypes.data_as(c_double_p), self.N))

    def association_log(self, path):
        """CSV log of every data_association() decision from now on (None closes it): call, index, x, y, landmark
        (-1 = dropped), min_distance, runner_up, created - what the reference only prints (ekf_slam.cpp:290-329)."""
        check(self._L.ekf_association_log_open(self._h, None if path is None else str(path).encode()))

    def sigma_rows(self, rows):
        """Selected rows of the covariance, shape [len(rows), N] (maps too large to read back whole)."""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        out = np.zeros((rows.size, self.N))
        if rows.size:
            check(self._L.ekf_get_sigma_rows(self._h, rows.ctypes.data_as(_lib.c_i64_p), int(rows.size),
                                             out.ctypes.data_as(c_double_p), self.N))
        return out

    @property
    def sigma_diag(self):
        out = np.zeros(self.N)
        check(self._L.ekf_get_sigma_diag(self._h, out.ctypes.data_as(c_double_p)))
        return out

    @property
    def init_flag(self):
        v = ctypes.c_int()
        check(self._L.ekf_get_init_flag(self._h, ctypes.byref(v)))
        return bool(v.value)

    @init_flag.setter
    def init_flag(self, v):
        check(self._L.ekf_set_init_flag(self._h, int(bool(v))))

    @property
    def update_count(self):
        v = ctypes.c_uint64()
        check(self._L.ekf_update_count(self._h, ctypes.byref(v)))
        return v.value

    @property
    def launch_count(self):
        v = ctypes.c_uint64()
        check(self._L.ekf_launch_count(self._h, ctypes.byref(v)))
        return v.value

    def sync(self):
        check(self._L.ekf_sync(self._h))

    @property
    def sweep_count(self):
        v = ctypes.c_uint64()
        check(self._L.ekf_sweep_count(self._h, ctypes.byref(v)))
        return v.value

    def set_max_pending(self, k):
        """Streamed engine: corrections accumulated per pass over Sigma (1..20, default 14); results do not depend on it."""
        check(self._L.ekf_set_max_pending(self._h, int(k)))

    def set_carry_pending(self, on):
        """Streamed engine: let correction factors stay pending across prediction() / measurement() calls (default on;
        off = Sigma is swept at the end of every measurement(), bit-identical to one sweep per correction)."""
        check(self._L.ekf_set_carry_pending(self._h, 1 if on else 0))

    def timer_start(self):
        check(self._L.ekf_timer_start(self._h))

    def timer_stop(self):
        ms = ctypes.c_float()
        check(self._L.ekf_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def clone(self):
        other = object.__new__(EKF_SLAM)
        other._L, other.n, other.N, other.last_assoc = self._L, self.n, self.N, None
        other._pose_cache = None
        h = ctypes.c_void_p()
        check(self._L.ekf_clone(self._h, ctypes.byref(h)))
        other._h = h
        return other


class PinnedBuffer:
    """Page-locked host array from ekf_host_alloc (makes the batched verbs' copies asynchronous)."""

    def __init__(self, shape, dtype):
        self._L = _lib.load()
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = ctypes.c_void_p()
        check(self._L.ekf_host_alloc(ctypes.byref(p), nbytes))
        self._p = p
        buf = (ctypes.c_char * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    @property
    def ptr(self):
        return self._p.value

    def close(self):
        if getattr(self, "_p", None):
            self.array = None
            self._L.ekf_host_free(self._p)
            self._p = None

    __del__ = close


def _ptr(a, dtype=None, size=None, what="array"):
    """Address of a host buffer for the C ABI, which receives no lengths: numpy arrays (and PinnedBuffers) are checked
    for dtype, contiguity and element count here, because a wrong one would be read past its end or reinterpreted
    silently.  A raw integer address is passed through (the caller vouches for it)."""
    if isinstance(a, PinnedBuffer):
        a = a.array
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError(f"{what}: array must be C-contiguous")
        if dtype is not None and a.dtype != np.dtype(dtype):
            raise TypeError(f"{what}: expected dtype {np.dtype(dtype)}, got {a.dtype}")
        if size is not None and a.size < size:
            raise ValueError(f"{what}: expected at least {size} elements, got {a.size}")
        return a.ctypes.data
    return int(a)


def marker_list(xy, visible):
    """Dense fake-sensor arrays ([B,2n] readings, [B,n] visible flags) -> the marker list step_known_sparse() takes:
    (offsets [B+1] int32, ids [total] uint8, xy [total,2]); only visible markers are listed, in id order."""
    vis = np.asarray(visible) != 0
    B, n = vis.shape
    if n > 256:
        raise ValueError("marker ids are uint8: n <= 256")
    offsets = np.zeros(B + 1, dtype=np.int32)
    np.cumsum(vis.sum(axis=1), out=offsets[1:])
    rows, ids = np.nonzero(vis)
    pts = np.asarray(xy, dtype=np.float64).reshape(B, n, 2)[rows, ids]
    return offsets, ids.astype(np.uint8), np.ascontiguousarray(pts)


class EKFBatch:
    """B independent filters on one GPU (Monte-Carlo noise-seed sweep, SURVEY.md §8d cfg3).  Up to 64 landmarks the
    covariance stays on chip during a step (`engine` == ENGINE_FUSED); from 65 to 1,024 it lives in HBM and each filter
    is bit-identical to an EKF_SLAM(n, engine=ENGINE_STREAM) with set_carry_pending(False) (`engine` ==
    ENGINE_STREAM; unknown association is not available there)."""

    def __init__(self, n_filters, n_measurements=20, device=0):
        self._L = _lib.load()
        self.B = int(n_filters)
        self.n = int(n_measurements)
        self.N = 3 + 2 * self.n
        h = ctypes.c_void_p()
        check(self._L.ekf_batch_create(self.B, self.n, device, ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.ekf_batch_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def engine(self):
        """ENGINE_FUSED (covariance on chip, n <= 64) or ENGINE_STREAM (covariance in HBM, 64 < n <= 1024)."""
        return self._L.ekf_batch_engine(self._h)

    @property
    def sweep_count(self):
        """Passes over a filter's covariance in HBM so far, summed over the filters (0 for the on-chip engines)."""
        v = ctypes.c_uint64()
        check(self._L.ekf_batch_sweep_count(self._h, ctypes.byref(v)))
        return v.value

    def step_known(self, twists, xy, visible):
        """prediction + measurement for every filter; host arrays [B,2], [B,2n], [B,n] (uint8)."""
        B, n = self.B, self.n
        check(self._L.ekf_batch_step_known(self._h, _ptr(twists, np.float64, 2 * B, "twists"),
                                           _ptr(xy, np.float64, 2 * n * B, "xy"), _ptr(visible, np.uint8, n * B, "visible")))

    def step_known_sparse(self, twists, offsets, ids, xy, total=None):
        """prediction + measurement from the marker list (visible markers only): twists [B,2], CSR offsets [B+1] int32,
        ids [total] uint8, xy [total,2].  Bit-identical to step_known() on the dense arrays (unlisted slots = 0)."""
        if isinstance(offsets, (np.ndarray, PinnedBuffer)):
            off = offsets.array if isinstance(offsets, PinnedBuffer) else offsets
            last = int(off.reshape(-1)[self.B])
            if total is not None and int(total) != last:
                raise ValueError(f"total = {total} does not match offsets[B] = {last}")
            total = last
        elif total is None:
            raise ValueError("total is required when offsets is a raw address")
        total = int(total)
        check(self._L.ekf_batch_step_known_sparse(self._h, _ptr(twists, np.float64, 2 * self.B, "twists"),
                                                  _ptr(offsets, np.int32, self.B + 1, "offsets"),
                                                  _ptr(ids, np.uint8, total, "ids"), _ptr(xy, np.float64, 2 * total, "xy"),
                                                  total))

    def step_unknown(self, twists, meas, count, m_max, want_assoc=False):
        """prediction + data_association; host arrays [B,2], [B,m_max,2], [B] int32."""
        assoc = np.empty((self.B, m_max), dtype=np.int32) if want_assoc else None
        check(self._L.ekf_batch_step_unknown(self._h, _ptr(twists, np.float64, 2 * self.B, "twists"),
                                             _ptr(meas, np.float64, 2 * int(m_max) * self.B, "meas"),
                                             _ptr(count, np.int32, self.B, "count"), int(m_max),
                                             assoc.ctypes.data if want_assoc else None))
        return assoc

    def step_known_dev(self, d_twists, d_xy, d_visible):
        check(self._L.ekf_batch_step_known_dev(self._h, int(d_twists), int(d_xy), int(d_visible)))

    def step_unknown_dev(self, d_twists, d_meas, d_count, m_max, d_assoc=None):
        check(self._L.ekf_batch_step_unknown_dev(self._h, int(d_twists), int(d_meas), int(d_count) if d_count else None,
                                                 int(m_max), int(d_assoc) if d_assoc else None))

    def poses(self):
        out = np.empty((self.B, 3))
        check(self._L.ekf_batch_get_poses(self._h, out.ctypes.data))
        return out

    def poses_async(self, pinned):
        check(self._L.ekf_batch_get_poses_async(self._h, _ptr(pinned, np.float64, 3 * self.B, "poses")))

    def states(self):
        out = np.empty((self.B, self.N))
        check(self._L.ekf_batch_get_states(self._h, out.ctypes.data_as(c_double_p)))
        return out

    def sigma(self, filt):
        out = np.empty((self.N, self.N))
        check(self._L.ekf_batch_get_sigma(self._h, int(filt), out.ctypes.data_as(c_double_p), self.N))
        return out

    @property
    def known(self):
        out = np.empty((self.B, self.n), dtype=np.uint8)
        check(self._L.ekf_batch_get_known(self._h, out.ctypes.data_as(c_u8_p)))
        return out

    @known.setter
    def known(self, v):
        v = np.ascontiguousarray(v, dtype=np.uint8)
        assert v.shape == (self.B, self.n)
        check(self._L.ekf_batch_set_known(self._h, v.ctypes.data_as(c_u8_p)))

    @property
    def update_count(self):
        v = ctypes.c_uint64()
        check(self._L.ekf_batch_update_count(self._h, ctypes.byref(v)))
        return v.value

    @property
    def launch_count(self):
        v = ctypes.c_uint64()
        check(self._L.ekf_batch_launch_count(self._h, ctypes.byref(v)))
        return v.value

    def pose_error(self, truth_xyt):
        """Per-GPU partial error statistics {sum dx^2, sum dy^2, sum dtheta^2, count} (the only thing ranks exchange)."""
        t = np.ascontiguousarray(truth_xyt, dtype=np.float64)
        assert t.shape == (self.B, 3)
        out = np.zeros(4)
        check(self._L.ekf_batch_pose_error(self._h, t.ctypes.data_as(c_double_p), out.ctypes.data_as(c_double_p)))
        return out

    # --- consistency (no reference counterpart; read on the device, in the engine's layout)
    def marginals(self):
        """(pose [B,3,3] in state order theta, x, y; landmarks [B,n,2,2]), both symmetric: the stored entries of
        sigma(b), bit for bit, without pulling whole covariances to the host."""
        pc = np.empty((self.B, 6))
        lc = np.empty((self.B, self.n, 3))
        check(self._L.ekf_batch_get_marginals(self._h, pc.ctypes.data, lc.ctypes.data))
        pose = pc[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(self.B, 3, 3)
        lm = lc[:, :, [0, 1, 1, 2]].reshape(self.B, self.n, 2, 2)
        return pose, lm

    def _lm_stride(self, shape):
        if shape == (self.n, 2):
            return 0
        if shape == (self.B, self.n, 2):
            return 2 * self.n
        raise ValueError(f"lm_truth must be [n,2] or [B,n,2], got {shape}")

    def nees(self, truth_xyt, lm_truth=None, per_filter=False):
        """Normalised estimation error squared of every filter against truth [B,3] = (x, y, theta) and, optionally,
        landmark truth [n,2] (shared by every filter) or [B,n,2]; NaN entries are not scored.  A landmark slot is scored
        once the filter has initialised it (first measurement(), or known[b, i] on the association path).  Returns
        consistency.anees_from_stats() of the batch partial, the partial itself as "stats" (additive: multi-GPU runs
        sum it with sharding.allreduce_sum), and with per_filter the arrays "pose_nees" [B] (NaN where not scored),
        "landmark_nees_sum" [B] and "landmark_nees_count" [B]."""
        from .consistency import anees_from_stats
        t = np.ascontiguousarray(truth_xyt, dtype=np.float64)
        if t.shape != (self.B, 3):
            raise ValueError(f"truth must be [B,3], got {t.shape}")
        lm = stride = None
        if lm_truth is not None:
            lm = np.ascontiguousarray(lm_truth, dtype=np.float64)
            stride = self._lm_stride(lm.shape)
        pf = np.empty((self.B, 3)) if per_filter else None
        out = np.zeros(8)
        check(self._L.ekf_batch_nees(self._h, t.ctypes.data, lm.ctypes.data if lm is not None else None, stride or 0,
                                     pf.ctypes.data if per_filter else None, out.ctypes.data))
        res = anees_from_stats(out)
        res["stats"] = out
        if per_filter:
            res["pose_nees"], res["landmark_nees_sum"], res["landmark_nees_count"] = pf[:, 0], pf[:, 1], pf[:, 2]
        return res

    def nees_dev(self, d_truth, d_out8, d_lm_truth=None, lm_truth_stride=0, d_per_filter=None):
        """ekf_batch_nees_dev: the same read-out from device pointers (truth [B][3], landmark truth [n][2] with stride 0
        or [B][n][2] with stride 2n, per-filter [B][3], out8 [8]), enqueued on the batch's stream without a
        synchronisation; the results are valid after sync()."""
        check(self._L.ekf_batch_nees_dev(self._h, int(d_truth) if d_truth else None, int(d_lm_truth) if d_lm_truth else None,
                                         int(lm_truth_stride), int(d_per_filter) if d_per_filter else None,
                                         int(d_out8) if d_out8 else None))

    def set_nis(self, on=True):
        """ekf_batch_set_nis: with on, the following steps also accumulate every filter's normalised innovation squared
        (NIS = nu^T S^-1 nu of each scored correction; the accumulators are allocated and zeroed on first use); with
        off, the plain step kernels run again and the accumulators are kept.  Checkpoints do not carry them."""
        check(self._L.ekf_batch_set_nis(self._h, 1 if on else 0))

    def nis(self, per_filter=False, reset=False):
        """NIS read-out, the consistency test that needs no truth: consistency.anis_from_stats() of the batch total
        {sum NIS, sum NIS^2, #scored, #non-finite} (also returned as "stats"; additive across ranks), and with
        per_filter the arrays "nis_sum", "nis_sq_sum", "nis_count" and "nis_nonfinite" [B].  reset zeroes the
        accumulators after the read.  Raises before set_nis() was ever called."""
        from .consistency import anis_from_stats
        pf = np.empty((self.B, 4)) if per_filter else None
        out = np.zeros(4)
        check(self._L.ekf_batch_nis(self._h, pf.ctypes.data if per_filter else None, out.ctypes.data, 1 if reset else 0))
        res = anis_from_stats(out)
        res["stats"] = out
        if per_filter:
            res["nis_sum"], res["nis_sq_sum"], res["nis_count"], res["nis_nonfinite"] = pf[:, 0], pf[:, 1], pf[:, 2], pf[:, 3]
        return res

    def nis_dev(self, d_out4, d_per_filter=None, reset=False):
        """ekf_batch_nis_dev: the same read-out into device pointers (out4 [4], per-filter [B][4]), enqueued on the
        batch's stream without a synchronisation; the results are valid after sync()."""
        check(self._L.ekf_batch_nis_dev(self._h, int(d_per_filter) if d_per_filter else None,
                                        int(d_out4) if d_out4 else None, 1 if reset else 0))

    def sync(self):
        check(self._L.ekf_batch_sync(self._h))

    def timer_start(self):
        check(self._L.ekf_batch_timer_start(self._h))

    def timer_stop(self):
        ms = ctypes.c_float()
        check(self._L.ekf_batch_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def checkpoint(self):
        """Everything needed to resume the batch bit-identically (dict of numpy arrays; Sigma in the engine's own layout,
        see device_pointers).  save_checkpoint / load_checkpoint put it in an .npz file."""
        ns, nst = ctypes.c_int64(), ctypes.c_int64()
        check(self._L.ekf_batch_checkpoint_size(self._h, ctypes.byref(ns), ctypes.byref(nst)))
        ck = {"sigma_packed": np.empty(ns.value), "state": np.empty(nst.value),
              "init_flag": np.empty(self.B, dtype=np.int32), "known": np.empty((self.B, self.n), dtype=np.uint8)}
        upd = ctypes.c_uint64()
        check(self._L.ekf_batch_export(self._h, ck["sigma_packed"].ctypes.data, ck["state"].ctypes.data,
                                       ck["init_flag"].ctypes.data, ck["known"].ctypes.data, ctypes.byref(upd)))
        ck["updates"] = np.uint64(upd.value)
        ck["shape"] = np.array([self.B, self.n], dtype=np.int64)
        return ck

    def restore(self, ck):
        if tuple(int(v) for v in ck["shape"]) != (self.B, self.n):
            raise ValueError("checkpoint is for a batch of another shape")
        ns, nst = ctypes.c_int64(), ctypes.c_int64()
        check(self._L.ekf_batch_checkpoint_size(self._h, ctypes.byref(ns), ctypes.byref(nst)))
        sig = np.ascontiguousarray(ck["sigma_packed"], dtype=np.float64)
        st = np.ascontiguousarray(ck["state"], dtype=np.float64)
        fl = np.ascontiguousarray(ck["init_flag"], dtype=np.int32)
        kn = np.ascontiguousarray(ck["known"], dtype=np.uint8)
        if sig.size != ns.value or st.size != nst.value or fl.size != self.B or kn.size != self.B * self.n:
            raise ValueError("checkpoint arrays do not match this build's layout")
        check(self._L.ekf_batch_import(self._h, sig.ctypes.data, st.ctypes.data, fl.ctypes.data, kn.ctypes.data,
                                       int(ck["updates"])))

    def save_checkpoint(self, path):
        np.savez(path, **self.checkpoint())

    def load_checkpoint(self, path):
        with np.load(path) as z:
            self.restore({k: z[k] for k in z.files})

    def device_pointers(self):
        """(sigma, sigma_stride, state, state_stride): device addresses and per-filter strides in doubles.  Sigma is in
        the engine's layout: tile (n = 20), packed symmetric staircase (n <= 64), or dense N x ld rows with
        ld = N rounded up to 16 (n > 64, sigma_stride = N * ld)."""
        s, st = ctypes.c_void_p(), ctypes.c_void_p()
        ss, sts = ctypes.c_int64(), ctypes.c_int64()
        check(self._L.ekf_batch_device_pointers(self._h, ctypes.byref(s), ctypes.byref(ss), ctypes.byref(st),
                                                ctypes.byref(sts)))
        return s.value, ss.value, st.value, sts.value

    @property
    def stream(self):
        return self._L.ekf_batch_stream(self._h)
