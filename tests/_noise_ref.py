"""Reference EKF-SLAM with per-filter noise covariances (test infrastructure only).

A numpy restatement of oracle/ekf_oracle.c in which Q = diag(q_theta, q_x, q_y) and R = diag(r_range, r_bearing) are
arguments instead of the reference's constants (1e-4 and 0.01).  Every product and sum is formed in the oracle's
order with one rounding each (numpy elementwise operations, Python floats, and the C library's sqrt / atan2 / sin /
cos / fmod through the math module), so with the reference values it is bit-identical to the oracle;
tests/test_noise_cpu.py pins that.  It also accumulates the NIS of the corrections that the batch engines score
(consistency.anis_from_stats' {sum, sum^2, #scored, #non-finite}).
"""
import math

import numpy as np

DEFAULT_NOISE = (1e-4, 1e-4, 1e-4, 0.01, 0.01)


def normalize_angle(rad):  # oracle_normalize_angle, rigid2d.cpp:336-345
    reduced = math.fmod(rad, 2 * math.pi)
    ang = math.fmod(reduced + 2 * math.pi, 2 * math.pi)
    return ang - 2 * math.pi if ang > math.pi else ang


class NoiseOracle:
    def __init__(self, n, noise=DEFAULT_NOISE):
        self.n, self.N = int(n), 3 + 2 * int(n)
        self.state = np.zeros(self.N)
        self.sigma = np.zeros((self.N, self.N))
        self.sigma[np.arange(3, self.N), np.arange(3, self.N)] = 100.0
        self.init_flag = False
        self.acc = np.zeros(4)
        self.values = []  # every scored value, in order
        self.set_noise(noise)

    def set_noise(self, noise):
        self.q = [float(v) for v in noise[:3]]
        self.r = [float(v) for v in noise[3:5]]

    # ekf_slam.cpp:55-106
    def prediction(self, dtheta, dx):
        dtheta, dx = float(dtheta), float(dx)
        s, th = self.sigma, float(self.state[0])
        if abs(dtheta) < 0.000001:
            u0, u1, u2 = 0.0, dx * math.cos(th), dx * math.sin(th)
            a1, a2 = -dx * math.sin(th), dx * math.cos(th)
        else:
            q = dx / dtheta
            u0 = dtheta
            u1 = -q * math.sin(th) + q * math.sin(th + dtheta)
            u2 = q * math.cos(th) - q * math.cos(th + dtheta)
            a1 = -q * math.cos(th) + q * math.cos(th + dtheta)
            a2 = -q * math.sin(th) + q * math.sin(th + dtheta)
        self.state[0] += u0
        self.state[1] += u1
        self.state[2] += u2
        s[1] = s[1] + a1 * s[0]
        s[2] = s[2] + a2 * s[0]
        c0 = s[:, 0].copy()
        s[:, 1] = s[:, 1] + c0 * a1
        s[:, 2] = s[:, 2] + c0 * a2
        for k in range(3):
            s[k, k] += self.q[k]

    def _h(self, i, theta, x, y):
        mx, my = float(self.state[3 + 2 * i]), float(self.state[4 + 2 * i])
        dx, dy = mx - x, my - y
        d = dx * dx + dy * dy
        zhat = (math.sqrt(dx * dx + dy * dy), normalize_angle(math.atan2(my - y, mx - x) - theta))
        H = ((0.0, -dx / math.sqrt(d), -dy / math.sqrt(d), dx / math.sqrt(d), dy / math.sqrt(d)),
             (-1.0, dy / d, -dx / d, -dy / d, dx / d))
        return H, zhat

    def _s_inverse(self, S):
        det = S[0][0] * S[1][1] - S[0][1] * S[1][0]
        return ((S[1][1] / det, -S[0][1] / det), (-S[1][0] / det, S[0][0] / det))

    def innovation_covariance(self, i, theta, x, y):
        """S = H Sigma H^T + R of landmark i at the pose (theta, x, y), in the correction's summation order."""
        H, _ = self._h(i, theta, x, y)
        idx = (0, 1, 2, 3 + 2 * i, 4 + 2 * i)
        W = [sum_rows(H[a], [self.sigma[k] for k in idx]) for a in range(2)]
        return [[sum_terms([W[a][idx[k]] * H[b][k] for k in range(5)]) + (self.r[a] if a == b else 0.0)
                 for b in range(2)] for a in range(2)], W, H

    # ekf_slam.cpp:138-192
    def _correct(self, i, sx, sy, theta, x, y, score):
        S, W, H = self.innovation_covariance(i, theta, x, y)
        _, zhat = self._h(i, theta, x, y)
        idx = (0, 1, 2, 3 + 2 * i, 4 + 2 * i)
        P = [sum_rows(H[a], [self.sigma[:, k] for k in idx]) for a in range(2)]
        Si = self._s_inverse(S)
        K0 = P[0] * Si[0][0] + P[1] * Si[1][0]
        K1 = P[0] * Si[0][1] + P[1] * Si[1][1]
        nu0 = math.sqrt(sx * sx + sy * sy) - zhat[0]
        nu1 = normalize_angle(math.atan2(sy, sx) - zhat[1])
        self.state = self.state + (K0 * nu0 + K1 * nu1)
        self.state[0] = normalize_angle(float(self.state[0]))
        self.sigma = self.sigma - (np.outer(K0, W[0]) + np.outer(K1, W[1]))
        if score:
            t0 = Si[0][0] * nu0 + Si[1][0] * nu1
            t1 = Si[0][1] * nu0 + Si[1][1] * nu1
            v = nu0 * t0 + nu1 * t1
            if math.isfinite(v):
                self.acc += (v, v * v, 1.0, 0.0)
                self.values.append(v)
            else:
                self.acc[3] += 1.0

    def _init_landmark(self, i, sx, sy, theta, x, y):
        ri, phii = math.sqrt(sx * sx + sy * sy), math.atan2(sy, sx)
        self.state[3 + 2 * i] = x + ri * math.cos(phii + theta)
        self.state[4 + 2 * i] = y + ri * math.sin(phii + theta)

    # ekf_slam.cpp:108-197
    def measurement(self, xy, visible):
        xy = np.asarray(xy, dtype=np.float64).reshape(-1)
        theta, x, y = (float(v) for v in self.state[:3])
        score = self.init_flag
        if not self.init_flag:
            for i in range(self.n):
                self._init_landmark(i, float(xy[2 * i]), float(xy[2 * i + 1]), theta, x, y)
            self.init_flag = True
        for i in range(self.n):
            if visible[i]:
                self._correct(i, float(xy[2 * i]), float(xy[2 * i + 1]), theta, x, y, score)

    # ekf_slam.cpp:217-276 (bearing innovation not wrapped)
    def maha(self, sx, sy, i):
        theta, x, y = (float(v) for v in self.state[:3])
        H, zhat = self._h(i, theta, x, y)
        idx = (0, 1, 2, 3 + 2 * i, 4 + 2 * i)
        Wl = [[sum_terms([H[a][k] * float(self.sigma[idx[k], idx[l]]) for k in range(5)]) for l in range(5)]
              for a in range(2)]
        psi = [[sum_terms([Wl[a][l] * H[b][l] for l in range(5)]) + (self.r[a] if a == b else 0.0) for b in range(2)]
               for a in range(2)]
        pi = self._s_inverse(psi)
        v0 = math.sqrt(sx * sx + sy * sy) - zhat[0]
        v1 = math.atan2(sy, sx) - zhat[1]
        t0 = v0 * pi[0][0] + v1 * pi[1][0]
        t1 = v0 * pi[0][1] + v1 * pi[1][1]
        return t0 * v0 + t1 * v1

    # ekf_slam.cpp:278-402; known updated in place; returns (assoc, created)
    def data_association(self, meas, known):
        meas = np.asarray(meas, dtype=np.float64).reshape(-1, 2)
        kc = 0
        while kc < self.n and known[kc]:
            kc += 1
        assoc = np.full(len(meas), -1, np.int32)
        created = np.zeros(len(meas), np.uint8)
        for j, (sx, sy) in enumerate(meas):
            sx, sy = float(sx), float(sy)
            min_d, min_idx = 10.0, kc
            for i in range(kc):
                d = self.maha(sx, sy, i)
                if d < min_d:
                    min_d, min_idx = d, i
            new = min_idx == kc and min_idx < self.n
            if new:
                self._init_landmark(min_idx, sx, sy, *(float(v) for v in self.state[:3]))
                known[kc] = 1
                kc += 1
                min_d = 0.0
                created[j] = 1
            if min_d < 1.0:
                self._correct(min_idx, sx, sy, *(float(v) for v in self.state[:3]), score=not new)
                assoc[j] = min_idx
        return assoc, created


def sum_terms(terms):
    acc = 0.0
    for t in terms:
        acc += t
    return acc


def sum_rows(h, rows):
    """sum_k h[k] * rows[k] over five rows, accumulated from 0.0 in index order (elementwise)."""
    acc = 0.0
    for hk, row in zip(h, rows):
        acc = acc + hk * row
    return acc
