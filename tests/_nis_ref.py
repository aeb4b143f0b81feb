"""Reference NIS (normalised innovation squared) of the CPU oracle's filter, for the batch engines' NIS variants.

NisOracle drives an OracleEKF and, before each measurement() / data_association() call, replays that call's corrections
in numpy from the oracle's own state and Sigma (the arithmetic of correct_landmark in oracle/ekf_oracle.c), keeping
    S = H_j Sigma H_j^T + R,  nu = (z_r - zhat_r, wrap(z_phi - zhat_phi)),  NIS = nu^T S^-1 nu
of every correction under the rule of ekf_batch_set_nis: a filter's first measurement() call scores nothing, a
landmark created by the reading it is corrected with is not scored, a dropped reading is no correction.  The replayed
state is checked against the oracle's after every call, so the S and nu are those the oracle used.
Accumulators: {sum NIS, sum NIS^2, #scored, #non-finite}, summed per call in correction order and then added, like
the kernels do."""
import math

import numpy as np

from _oracle import OracleEKF

R = 0.01


def wrap(a):
    """oracle_normalize_angle: (-pi, pi] through two fmods"""
    red = math.fmod(a, 2 * math.pi)
    ang = math.fmod(red + 2 * math.pi, 2 * math.pi)
    return ang - 2 * math.pi if ang > math.pi else ang


def nis_value(si, nu0, nu1):
    """nu0 (i00 nu0 + i10 nu1) + nu1 (i01 nu0 + i11 nu1), each operation rounded on its own (ekf_math.cuh nis())"""
    return nu0 * (si[0][0] * nu0 + si[1][0] * nu1) + nu1 * (si[0][1] * nu0 + si[1][1] * nu1)


class NisOracle:
    def __init__(self, n):
        self.o = OracleEKF(n)
        self.n, self.N = n, 3 + 2 * n
        self.acc = np.zeros(4)
        self.values = []  # every scored value, in order

    def prediction(self, dtheta, dx):
        self.o.prediction(dtheta, dx)

    def _correct(self, st, P, i, sx, sy, theta, x, y):
        """correct_landmark on (st, P) in place; returns NIS"""
        mx, my = st[3 + 2 * i], st[4 + 2 * i]
        dx, dy = mx - x, my - y
        d = dx * dx + dy * dy
        q = math.sqrt(d)
        zhat = (q, wrap(math.atan2(dy, dx) - theta))
        idx = [0, 1, 2, 3 + 2 * i, 4 + 2 * i]
        H = np.array([[0.0, -dx / q, -dy / q, dx / q, dy / q], [-1.0, dy / d, -dx / d, -dy / d, dx / d]])
        W = H @ P[idx, :]
        S = W[:, idx] @ H.T + R * np.eye(2)
        det = S[0, 0] * S[1, 1] - S[0, 1] * S[1, 0]
        si = [[S[1, 1] / det, -S[0, 1] / det], [-S[1, 0] / det, S[0, 0] / det]]
        K = W.T @ np.array(si)
        nu0 = math.sqrt(sx * sx + sy * sy) - zhat[0]
        nu1 = wrap(math.atan2(sy, sx) - zhat[1])
        st += K @ np.array([nu0, nu1])
        st[0] = wrap(st[0])
        P -= K @ W
        return nis_value(si, nu0, nu1)

    def _add(self, vals):
        step = np.zeros(4)
        for v in vals:
            if math.isfinite(v):
                step += (v, v * v, 1.0, 0.0)
                self.values.append(v)
            else:
                step[3] += 1.0
        self.acc += step

    def _check(self, st):
        ref = self.o.state
        err = np.max(np.abs(st - ref) / np.maximum(1.0, np.abs(ref)))
        assert err < 1e-9, f"numpy replay left the oracle's state: {err:.3e}"

    def measurement(self, xy, visible):
        xy = np.asarray(xy, dtype=np.float64).reshape(-1)
        vis = np.asarray(visible).reshape(-1)
        vals = []
        if self.o.init_flag:
            st, P = self.o.state, self.o.sigma
            theta, x, y = st[0], st[1], st[2]
            for i in range(self.n):
                if vis[i]:
                    vals.append(self._correct(st, P, i, xy[2 * i], xy[2 * i + 1], theta, x, y))
            self.o.measurement(xy, vis)
            self._check(st)
        else:
            self.o.measurement(xy, vis)
        self._add(vals)

    def data_association(self, xy, known):
        xy = np.asarray(xy, dtype=np.float64).reshape(-1)
        st, P = self.o.state, self.o.sigma
        out = self.o.data_association(xy, known)
        assoc, _, _, created = out
        vals = []
        for j in range(assoc.size):
            sx, sy = xy[2 * j], xy[2 * j + 1]
            if created[j]:
                i = assoc[j]
                r, phi = math.sqrt(sx * sx + sy * sy), math.atan2(sy, sx)
                st[3 + 2 * i] = st[1] + r * math.cos(phi + st[0])
                st[4 + 2 * i] = st[2] + r * math.sin(phi + st[0])
            if assoc[j] >= 0:
                v = self._correct(st, P, int(assoc[j]), sx, sy, st[0], st[1], st[2])
                if not created[j]:
                    vals.append(v)
        self._check(st)
        self._add(vals)
        return out
