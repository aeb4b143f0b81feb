// Scalar building blocks of the EKF-SLAM hot path, shared by every engine (fused on-chip filter,
// streamed large map, row-sharded map).  fp64 throughout, to match the reference's Armadillo doubles.
//
// The geometry (z_hat, H_j, 2x2 inverse) is written with explicit round-to-nearest intrinsics so that
// nvcc does not contract a*b+c into an FMA there: the reference's x86-64 build rounds twice, and keeping
// the same rounding in the O(1) part of each update costs nothing.  The O(N) / O(N^2) parts use FMAs.
//
// Reference lines are relative to /root/reference/rigid2d/src/.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

// How the O(1) geometry of a correction forms its quotients (H_j entries, S^-1):
//   0: eight true IEEE divisions + an IEEE sqrt, exactly the reference's operations;
//   1: three reciprocals + eight multiplications (each quotient carries up to one extra ulp);
//   2 (default): additionally 1/sqrt(d) from rsqrt(), sqrt(d) = d * rsqrt(d), 1/d = rsqrt(d)^2 (<= ~4 ulp).
// The scalar chain is what bounds the fused kernel (12 resident filters per SM, each a serial fp64 dependency chain):
// on B200 level 1 is 14 % and level 2 is 20 % faster than level 0 on the 65,536-filter batch, and all parity tests
// hold unchanged at 1e-9 (observed deviations stay at the 1e-11 level set by atan2 and the 1e4 conditioning).
#ifndef EKF_RECIPROCAL_MULTIPLY
#define EKF_RECIPROCAL_MULTIPLY 2
#endif

namespace ekf {

constexpr double kPi = 3.14159265358979323846;  // rigid2d.hpp:13
constexpr double kTwoPi = 2.0 * kPi;
constexpr double kR = 0.01;      // measurement noise, ekf_slam.cpp:172-175
constexpr double kQ = 0.0001;    // process noise on (theta, x, y), ekf_slam.cpp:41-43
constexpr double kSigma0 = 100;  // initial landmark variance, ekf_slam.cpp:32
constexpr double kGateNew = 10.0;    // ekf_slam.cpp:293
constexpr double kGateUpdate = 1.0;  // ekf_slam.cpp:330
constexpr double kSmallTurn = 0.000001;  // ekf_slam.cpp:79

// Process and measurement noise of one filter: Q = diag(q0, q1, q2) on (theta, x, y), R = diag(r0, r1) on (range,
// bearing).  ref_noise() holds the reference's constants; the default kernels pass it, so they compile as before, and
// the NOISE variants read a per-filter row {q_theta, q_x, q_y, r_range, r_bearing} (ekf_set_noise,
// ekf_batch_set_noise).
struct Noise {
    double q0, q1, q2, r0, r1;
};
__host__ __device__ constexpr Noise ref_noise() { return Noise{kQ, kQ, kQ, kR, kR}; }
__device__ __forceinline__ Noise load_noise(const double* __restrict__ row) {
    return Noise{row[0], row[1], row[2], row[3], row[4]};
}

// fmod(x, 2*pi), exact like the C library's: the quotient is small on this path, so one FMA recovers the
// remainder exactly (x and q*2pi are both multiples of ulp(2pi) once |x| >= 2pi, and the remainder is
// below 8 so it fits 53 bits).  Falls back to fmod() for large or non-finite arguments.
static __device__ __noinline__ double fmod_2pi(double x) {
    const double y = kTwoPi;
    const double ax = fabs(x);
    if (ax < y) return x;
    if (!(ax < 1.0e6)) return fmod(x, y);
    double q = trunc(ax * (1.0 / kTwoPi));
    double r = fma(-q, y, ax);
    if (r < 0.0) {
        q -= 1.0;
        r = fma(-q, y, ax);
    } else if (r >= y) {
        q += 1.0;
        r = fma(-q, y, ax);
    }
    return copysign(r, x);
}

// rigid2d::normalize_angle, rigid2d.cpp:336-345 -> (-pi, pi]
//   reduced = fmod(rad, 2pi); ang = fmod(reduced + 2pi, 2pi); if (ang > pi) ang -= 2pi
// For |rad| < 2pi (every angle on this path: sums and differences of two wrapped angles) the first fmod is the
// identity and the second one reduces t = rad + 2pi in [0, 4pi): t - 2pi is exact there (Sterbenz), so the result is
// bit-identical to the library formulation without a division or a truncation.
static __device__ __noinline__ double normalize_angle_large(double rad) {  // |rad| >= 2pi: never on the hot path
    const double reduced = fmod_2pi(rad);
    double ang = fmod_2pi(__dadd_rn(reduced, kTwoPi));
    if (ang > kPi) ang = __dsub_rn(ang, kTwoPi);
    return ang;
}
__device__ __forceinline__ double normalize_angle(double rad) {
    if (!(fabs(rad) < kTwoPi)) return normalize_angle_large(rad);
    const double t = __dadd_rn(rad, kTwoPi);
    double ang = (t >= kTwoPi) ? __dsub_rn(t, kTwoPi) : t;
    if (ang > kPi) ang = __dsub_rn(ang, kTwoPi);
    return ang;
}

// Range / bearing of a robot-frame point (ekf_slam.cpp:140-146, 227-233, 338-344).
__device__ __forceinline__ void range_bearing(double sx, double sy, double& r, double& phi) {
    r = sqrt(__dadd_rn(__dmul_rn(sx, sx), __dmul_rn(sy, sy)));
    phi = atan2(sy, sx);
}

// World position of a landmark seen at robot-frame (sx, sy): ekf_slam.cpp:113-128, 200-214.
__device__ __forceinline__ void landmark_from_reading(double sx, double sy, double theta, double x, double y,
                                                      double& mx, double& my) {
    double r, phi;
    range_bearing(sx, sy, r, phi);
    double s, c;
    sincos(__dadd_rn(phi, theta), &s, &c);
    mx = __dadd_rn(x, __dmul_rn(r, c));
    my = __dadd_rn(y, __dmul_rn(r, s));
}

// The five non-zero columns {0,1,2,3+2i,4+2i} of H_j and the predicted measurement
// (ekf_slam.cpp:150-170).  h[0][0] == 0 and h[1][0] == -1 are implied and not stored:
//   row 0: [0, a, b, -a, -b]   a = -dx/sqrt(d), b = -dy/sqrt(d)
//   row 1: [-1, e, f, -e, -f]  e =  dy/d,       f = -dx/d
struct Hj {
    double a, b, e, f;
    double zr, zphi;  // z_hat
};

__device__ __forceinline__ Hj make_hj(double mx, double my, double theta, double x, double y) {
    Hj h;
    const double dx = __dsub_rn(mx, x), dy = __dsub_rn(my, y);
    const double d = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
#if EKF_RECIPROCAL_MULTIPLY >= 2
    const double isq = rsqrt(d), sq = __dmul_rn(d, isq), id = __dmul_rn(isq, isq);
#else
    const double sq = sqrt(d);
#endif
    h.zr = sq;
    h.zphi = normalize_angle(__dsub_rn(atan2(dy, dx), theta));
#if EKF_RECIPROCAL_MULTIPLY >= 2
    h.a = -__dmul_rn(dx, isq);
    h.b = -__dmul_rn(dy, isq);
    h.e = __dmul_rn(dy, id);
    h.f = -__dmul_rn(dx, id);
#elif EKF_RECIPROCAL_MULTIPLY
    const double isq = 1.0 / sq, id = 1.0 / d;
    h.a = -__dmul_rn(dx, isq);
    h.b = -__dmul_rn(dy, isq);
    h.e = __dmul_rn(dy, id);
    h.f = -__dmul_rn(dx, id);
#else
    h.a = -(dx / sq);
    h.b = -(dy / sq);
    h.e = dy / d;
    h.f = -(dx / d);
#endif
    return h;
}

// ---- innovation without an atan2 per correction (fused symmetric engine) -------------------------------------
// The reference forms nu = [z_r - zhat_r, normalize(z_phi - zhat_phi)] from two atan2 results
// (ekf_slam.cpp:140-146, :163-170, :182-183).  The wrapped bearing difference IS the angle between the measured
// direction u = (sx, sy) / |s| and the predicted direction p = R(-theta) (dx, dy) / sqrt(d), both in the robot frame:
//   sin(nu_phi) = p x u,  cos(nu_phi) = p . u.
// Innovations are small (sensor noise + prediction error), so asin(sin(nu_phi)) from a short odd series is exact to
// below one ulp for |sin| < 1/8; anything else (and a NaN) takes the reference's formulation, out of line.
struct Reading {
    double zr, ux, uy;  // range and unit direction of a robot-frame reading
};
__device__ __forceinline__ Reading make_reading(double sx, double sy) {
    Reading z;
    z.zr = sqrt(__dadd_rn(__dmul_rn(sx, sx), __dmul_rn(sy, sy)));
    const double inv = 1.0 / z.zr;
    z.ux = z.zr > 0.0 ? sx * inv : 1.0;  // atan2(0, 0) == 0
    z.uy = z.zr > 0.0 ? sy * inv : 0.0;
    return z;
}

static __device__ __noinline__ double bearing_innovation_reference(double dy, double dx, double theta, double uy, double ux) {
    const double zhat_phi = normalize_angle(__dsub_rn(atan2(dy, dx), theta));
    return normalize_angle(__dsub_rn(atan2(uy, ux), zhat_phi));
}

__device__ __forceinline__ double asin_small(double x) {  // |x| < 1/8: truncation error < 3e-19 relative
    const double x2 = x * x;
    double p = 12155.0 / 2490368.0;  // unused tail guard term keeps the last kept term's error negligible
    p = fma(p, x2, 6435.0 / 557056.0);
    p = fma(p, x2, 143.0 / 10240.0);
    p = fma(p, x2, 231.0 / 13312.0);
    p = fma(p, x2, 63.0 / 2816.0);
    p = fma(p, x2, 35.0 / 1152.0);
    p = fma(p, x2, 5.0 / 112.0);
    p = fma(p, x2, 3.0 / 40.0);
    p = fma(p, x2, 1.0 / 6.0);
    return fma(x * x2, p, x);
}

struct Innov {
    double a, b, e, f;  // H_j entries as in Hj
    double nu0, nu1;
};
// (sth, cth) = sincos(theta) of the pose the reference linearises about.
__device__ __forceinline__ Innov make_innov(double mx, double my, double theta, double sth, double cth, double x,
                                            double y, const Reading z) {
    Innov h;
    const double dx = __dsub_rn(mx, x), dy = __dsub_rn(my, y);
    const double d = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    const double isq = rsqrt(d), sq = __dmul_rn(d, isq), id = __dmul_rn(isq, isq);
    h.a = -__dmul_rn(dx, isq);
    h.b = -__dmul_rn(dy, isq);
    h.e = __dmul_rn(dy, id);
    h.f = -__dmul_rn(dx, id);
    h.nu0 = __dsub_rn(z.zr, sq);
    const double px = fma(sth, dy, cth * dx), py = fma(cth, dy, -(sth * dx));
    const double sn = fma(px, z.uy, -(py * z.ux)) * isq;
    const double cs = fma(px, z.ux, py * z.uy);
    if (cs > 0.0 && fabs(sn) < 0.125)
        h.nu1 = asin_small(sn);
    else
        h.nu1 = bearing_innovation_reference(dy, dx, theta, z.uy, z.ux);
    return h;
}

// Rows of H applied to five gathered values s0..s4 (values at indices 0,1,2,3+2i,4+2i).
template <class H>
__device__ __forceinline__ double h_row0(const H& h, double s1, double s2, double s3, double s4) {
    return fma(-h.b, s4, fma(-h.a, s3, fma(h.b, s2, h.a * s1)));
}
template <class H>
__device__ __forceinline__ double h_row1(const H& h, double s0, double s1, double s2, double s3, double s4) {
    return fma(-h.f, s4, fma(-h.e, s3, fma(h.f, s2, fma(h.e, s1, -s0))));
}

// Both rows at once from the two differences they share: row 0 = a (s1 - s3) + b (s2 - s4),
// row 1 = -s0 + e (s1 - s3) + f (s2 - s4).  Six operations and a dependency depth of three instead of nine and five
// (same algebra as h_row0 / h_row1, different rounding order; used by the batched kernel's scalar chain).
template <class H>
__device__ __forceinline__ void h_rows(const H& h, double s0, double s1, double s2, double s3, double s4, double& r0,
                                       double& r1) {
    const double d13 = s1 - s3, d24 = s2 - s4;
    r0 = fma(h.b, d24, h.a * d13);
    r1 = fma(h.f, d24, fma(h.e, d13, -s0));
}

struct Sym2 {
    double i00, i01, i10, i11;
};

// (S)^-1 with Armadillo's closed form for 2x2 ([d -b; -c a] / det); S = [s00 s01; s10 s11].
__device__ __forceinline__ Sym2 inv2x2(double s00, double s01, double s10, double s11) {
    const double det = __dsub_rn(__dmul_rn(s00, s11), __dmul_rn(s01, s10));
    Sym2 r;
#if EKF_RECIPROCAL_MULTIPLY
    const double idet = 1.0 / det;
    r.i00 = __dmul_rn(s11, idet);
    r.i01 = __dmul_rn(-s01, idet);
    r.i10 = __dmul_rn(-s10, idet);
    r.i11 = __dmul_rn(s00, idet);
#else
    r.i00 = s11 / det;
    r.i01 = -s01 / det;
    r.i10 = -s10 / det;
    r.i11 = s00 / det;
#endif
    return r;
}

// Normalised innovation squared nu^T S^-1 nu of one correction, from exactly the S^-1 and nu its gain uses (the batch
// engines' NIS variants).  Every product and sum is rounded on its own, so a host restatement without FMA contraction
// gives the same value from the same inputs.
__device__ __forceinline__ double nis(const Sym2& si, double nu0, double nu1) {
    const double t0 = __dadd_rn(__dmul_rn(si.i00, nu0), __dmul_rn(si.i10, nu1));
    const double t1 = __dadd_rn(__dmul_rn(si.i01, nu0), __dmul_rn(si.i11, nu1));
    return __dadd_rn(__dmul_rn(nu0, t0), __dmul_rn(nu1, t1));
}
// acc = {sum NIS, sum NIS^2, #scored, #non-finite}: a value that is not finite is counted in acc[3] only
__device__ __forceinline__ void nis_add(double* acc, double v) {
    if (isfinite(v)) {
        acc[0] = __dadd_rn(acc[0], v);
        acc[1] = __dadd_rn(acc[1], __dmul_rn(v, v));
        acc[2] += 1.0;
    } else {
        acc[3] += 1.0;
    }
}

// Mahalanobis distance of measurement (zr, zphi) to landmark i, from the 5x5 block Sigma[idx, idx]
// (ekf_slam.cpp:217-276).  The bearing innovation is NOT wrapped (:269).  `sig` may point to shared or
// global memory; ld is the row stride in doubles.
// `robot` points at row 0 of Sigma (rows 0..2 are read from it), `lm` at row 3+2i (rows 3+2i, 4+2i); both with
// row stride ld.  They are the same matrix on one GPU and two different buffers in the row-sharded engine.
__device__ __forceinline__ double maha_distance_rows(const double* __restrict__ robot, const double* __restrict__ lm,
                                                     int64_t ld, int i, double mx, double my, double zr, double zphi,
                                                     double theta, double x, double y, const Noise& nz) {
    const Hj h = make_hj(mx, my, theta, x, y);
    const int64_t id[5] = {0, 1, 2, 3 + 2 * (int64_t)i, 4 + 2 * (int64_t)i};
    double wl0[5], wl1[5];
#pragma unroll
    for (int l = 0; l < 5; ++l) {
        const double s0 = robot[id[l]];
        const double s1 = robot[ld + id[l]];
        const double s2 = robot[2 * ld + id[l]];
        const double s3 = lm[id[l]];
        const double s4 = lm[ld + id[l]];
        wl0[l] = h_row0(h, s1, s2, s3, s4);
        wl1[l] = h_row1(h, s0, s1, s2, s3, s4);
    }
    // psi = (H Sigma) H^T + R
    const double p00 = h_row0(h, wl0[1], wl0[2], wl0[3], wl0[4]) + nz.r0;
    const double p01 = h_row1(h, wl0[0], wl0[1], wl0[2], wl0[3], wl0[4]);
    const double p10 = h_row0(h, wl1[1], wl1[2], wl1[3], wl1[4]);
    const double p11 = h_row1(h, wl1[0], wl1[1], wl1[2], wl1[3], wl1[4]) + nz.r1;
    const Sym2 pi = inv2x2(p00, p01, p10, p11);
    const double v0 = __dsub_rn(zr, h.zr), v1 = __dsub_rn(zphi, h.zphi);
    const double t0 = __dadd_rn(__dmul_rn(v0, pi.i00), __dmul_rn(v1, pi.i10));
    const double t1 = __dadd_rn(__dmul_rn(v0, pi.i01), __dmul_rn(v1, pi.i11));
    return __dadd_rn(__dmul_rn(t0, v0), __dmul_rn(t1, v1));
}

// Whole Sigma in one buffer (shared memory in the fused engine, global memory in the streamed one).
__device__ __forceinline__ double maha_distance(const double* __restrict__ sig, int64_t ld, int i, double mx,
                                                double my, double zr, double zphi, double theta, double x,
                                                double y, const Noise& nz) {
    return maha_distance_rows(sig, sig + (3 + 2 * (int64_t)i) * ld, ld, i, mx, my, zr, zphi, theta, x, y, nz);
}

// + Q on the robot block's diagonal after the motion Jacobian (ekf_slam.cpp:41-43, :102); s = rows 0..2, columns 0..2
__device__ __forceinline__ void add_process_noise(double (&s)[3][3], const Noise& nz) {
    s[0][0] += nz.q0;
    s[1][1] += nz.q1;
    s[2][2] += nz.q2;
}

// Motion model increments and Jacobian entries (ekf_slam.cpp:67-96): state[0..2] += u, A(1,0)=a1, A(2,0)=a2.
struct Motion {
    double u0, u1, u2, a1, a2;
    double s_new, c_new;  // sincos(theta + u0)
};
__device__ __forceinline__ Motion motion_model(double theta, double dtheta, double dx) {
    Motion m;
    double s, c;
    sincos(theta, &s, &c);
    if (fabs(dtheta) < kSmallTurn) {
        m.u0 = 0.0;
        m.u1 = __dmul_rn(dx, c);
        m.u2 = __dmul_rn(dx, s);
        m.a1 = __dmul_rn(-dx, s);
        m.a2 = __dmul_rn(dx, c);
        m.s_new = s;
        m.c_new = c;
    } else {
        double s2, c2;
        sincos(__dadd_rn(theta, dtheta), &s2, &c2);
        const double q = dx / dtheta;
        m.u0 = dtheta;
        m.u1 = __dadd_rn(__dmul_rn(-q, s), __dmul_rn(q, s2));
        m.u2 = __dsub_rn(__dmul_rn(q, c), __dmul_rn(q, c2));
        m.a1 = __dadd_rn(__dmul_rn(-q, c), __dmul_rn(q, c2));
        m.a2 = __dadd_rn(__dmul_rn(-q, s), __dmul_rn(q, s2));
        m.s_new = s2;
        m.c_new = c2;
    }
    return m;
}

// ---- dead-reckoning odometry (DiffDrive::updatePose, rigid2d/src/diff_drive.cpp:50-67) --------------------------
// Transform2D::operator*=, rigid2d.cpp:222-245: the composed rotation goes through acos / asin, kept as written.
__device__ __forceinline__ void compose_tf(double ax, double ay, double ath, double bx, double by, double bth,
                                           double& ox, double& oy, double& oth) {
    double sa, ca, sb, cb;
    sincos(ath, &sa, &ca);
    sincos(bth, &sb, &cb);
    const double r11 = __dsub_rn(__dmul_rn(ca, cb), __dmul_rn(sa, sb));
    const double r21 = __dadd_rn(__dmul_rn(sa, cb), __dmul_rn(ca, sb));
    const double rc = acos(r11), rs = asin(r21);
    oth = (__dmul_rn(rc, rs) < 0) ? rs : rc;
    ox = __dadd_rn(__dsub_rn(__dmul_rn(bx, ca), __dmul_rn(by, sa)), ax);
    oy = __dadd_rn(__dadd_rn(__dmul_rn(bx, sa), __dmul_rn(by, ca)), ay);
}
// integrateTwist, rigid2d.cpp:304-333
__device__ __forceinline__ void integrate_twist(double w, double vx, double vy, double& tx, double& ty, double& tth) {
    if (fabs(w) > 0.0001) {
        const double xs = vy / w, ys = -vx / w;
        double t1x, t1y, t1th;
        compose_tf(0.0, 0.0, w, xs, ys, 0.0, t1x, t1y, t1th);  // Transform2D(w) * Transform2D(p_sb)
        compose_tf(-xs, -ys, -0.0, t1x, t1y, t1th, tx, ty, tth);  // t_sb.inv() * (...)
    } else {
        tx = vx, ty = vy, tth = 0.0;
    }
}
// pose = {x, y, theta} in place; theta is not wrapped
__device__ __forceinline__ void update_pose(double wheel_base, double wheel_radius, double left, double right, double& x,
                                            double& y, double& theta) {
    const double D = __dmul_rn(wheel_base, 0.5), r = wheel_radius;
    const double w = __dmul_rn(r / __dmul_rn(2.0, D), __dsub_rn(right, left));
    const double vx = __dmul_rn(r / 2.0, __dadd_rn(right, left));
    double tx, ty, tth;
    integrate_twist(w, vx, 0.0, tx, ty, tth);
    double s, c;
    sincos(theta, &s, &c);
    x = __dadd_rn(x, __dsub_rn(__dmul_rn(tx, c), __dmul_rn(ty, s)));
    y = __dadd_rn(y, __dadd_rn(__dmul_rn(tx, s), __dmul_rn(ty, c)));
    theta = __dadd_rn(theta, tth);
}

// Lexicographic (distance, index) minimum used by the association argmin: strict '<' on distance,
// lowest index on ties (ekf_slam.cpp:300-309).  NaNs must be mapped to +inf by the caller.
__device__ __forceinline__ bool better(double d_a, int i_a, double d_b, int i_b) {
    return (d_a < d_b) || (d_a == d_b && i_a < i_b);
}

}  // namespace ekf
