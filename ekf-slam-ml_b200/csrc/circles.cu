// Laser landmark detection, batched over scans: rigid2d::CircleFitting
// (/root/reference/rigid2d/src/circle_fitting.cpp) re-designed for the GPU.
//   clusteringRanges  :11-90    one CTA per scan: parallel run detection, ordered compaction, wrap merge
//   circleRegression  :104-232  one warp per cluster: one-sided Jacobi SVD of the n x 4 design matrix held in
//                               registers, 4x4 symmetric Jacobi eigen-solve, closed-form solve through the SVD
//   classifyCircle    :234-296  same warp: mean inscribed angle + radius gate
// One kernel launch per batch of scans; nothing is computed on the host.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <new>

#include "../../include/circle_fit_b200.h"
#include "ekf_math.cuh"
#include "host_util.cuh"

namespace circ {

using ekf::kPi;
using ekf::kTwoPi;

constexpr int kMaxBeams = 384;  // 12 rows per lane; the reference's node uses 360 (landmarks.cpp:65)
constexpr int kRows = kMaxBeams / 32;
constexpr int kMaxClusters = 56;  // >= floor(383 / 7)
constexpr double kThresh = 0.2;   // circle_fitting.cpp:17
// One warp per scan, 16 scans resident per SM: measured on B200 (8,192 scans) 2.58 M scans/s, against 2.13 M with a
// 256-thread CTA per scan (the per-scan barriers leave seven warps waiting for the one with the wall cluster).
#ifndef CIRC_CTA_THREADS
#define CIRC_CTA_THREADS 32
#endif
#ifndef CIRC_MIN_CTAS
#define CIRC_MIN_CTAS 16
#endif
constexpr int kCtaThreads = CIRC_CTA_THREADS;

struct Segs {
    int s1, l1, s2, l2;  // points = beams s1..s1+l1-1 followed by s2..s2+l2-1
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// 4x4 symmetric eigen-decomposition by cyclic Jacobi.  q is destroyed (diagonal = eigenvalues), e = eigenvectors
// in columns.  Executed redundantly (and identically) by every lane.
__device__ __forceinline__ void jacobi_eig4(double q[4][4], double e[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) e[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 32; ++sweep) {
        double off = 0.0, diag = 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            diag += q[i][i] * q[i][i];
#pragma unroll
            for (int j = i + 1; j < 4; ++j) off += q[i][j] * q[i][j];
        }
        if (!(off > 1e-32 * diag)) break;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int r = p + 1; r < 4; ++r) {
                const double apq = q[p][r];
                if (fabs(apq) < 1e-300) continue;
                const double theta = (q[r][r] - q[p][p]) / (2.0 * apq);
                const double t = copysign(1.0, theta) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
                for (int k = 0; k < 4; ++k) {  // columns p, r
                    const double kp = q[k][p], kr = q[k][r];
                    q[k][p] = c * kp - s * kr;
                    q[k][r] = s * kp + c * kr;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {  // rows p, r
                    const double pk = q[p][k], rk = q[r][k];
                    q[p][k] = c * pk - s * rk;
                    q[r][k] = s * pk + c * rk;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double kp = e[k][p], kr = e[k][r];
                    e[k][p] = c * kp - s * kr;
                    e[k][r] = s * kp + c * kr;
                }
            }
        }
    }
}

struct FitResult {
    double cx, cy, r, mean_angle;
    int fallback;  // no eigenvalue in (0, 1000): the reference falls back to LAPACK's index 0 (unspecified order)
};

// Hyper-circle fit + inscribed-angle statistic of one cluster by one warp.  `pt(k)` returns point k.
// ROWS = design-matrix rows held per lane (cluster size <= 32 * ROWS): tube clusters have 7..40 points, so the
// common case runs with ROWS = 2 and a sixth of the register-array work of the general (ROWS = 12) instantiation.
// classifyCircle's statistic: mean inscribed angle over the interior points (:242-263)
template <class Fetch>
__device__ __forceinline__ double warp_mean_inscribed_angle(Fetch pt, const int n, const int lane) {
    const double2 p1 = pt(0), p2 = pt(n - 1);
    double sa = 0.0;
    for (int k = 1 + lane; k < n - 1; k += 32) {
        const double2 p = pt(k);
        const double ax = p1.x - p.x, ay = p1.y - p.y, bx = p2.x - p.x, by = p2.y - p.y;
        const double top = __dadd_rn(__dmul_rn(ax, bx), __dmul_rn(ay, by));
        const double bot = __dmul_rn(sqrt(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay))),
                                     sqrt(__dadd_rn(__dmul_rn(bx, bx), __dmul_rn(by, by))));
        sa += acos(top / bot);
    }
    return warp_sum(sa) / (double)(n - 2);
}
__device__ __forceinline__ bool angle_in_circle_range(double mean_angle) { return mean_angle > 1.5708 && mean_angle < 2.3562; }

template <int ROWS, class Fetch>
__device__ __forceinline__ FitResult warp_circle_fit_rows(Fetch pt, const int n, const int lane, const double mean_angle) {
    constexpr int kRows = ROWS;
    double a0[kRows], a1[kRows], a2[kRows], a3[kRows];
    // means (circle_fitting.cpp:112-120)
    double sx = 0.0, sy = 0.0;
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
        const int k = lane + 32 * j;
        double2 p = make_double2(0.0, 0.0);
        if (k < n) p = pt(k);
        a1[j] = p.x;
        a2[j] = p.y;
        sx += p.x;
        sy += p.y;
    }
    const double xm = warp_sum(sx) / (double)n, ym = warp_sum(sy) / (double)n;
    double sz = 0.0;
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
        const int k = lane + 32 * j;
        const bool v = k < n;
        const double x = v ? a1[j] - xm : 0.0, y = v ? a2[j] - ym : 0.0;
        a1[j] = x;
        a2[j] = y;
        a0[j] = x * x + y * y;
        a3[j] = v ? 1.0 : 0.0;
        sz += a0[j];
    }
    const double zm = warp_sum(sz) / (double)n;

    // one-sided Jacobi SVD of Z = [z x y 1]: rotate column pairs until mutually orthogonal; V accumulates
    double V[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
#define COL(c) ((c) == 0 ? a0 : (c) == 1 ? a1 : (c) == 2 ? a2 : a3)
    for (int sweep = 0; sweep < 40; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                double* cp = COL(p);
                double* cq = COL(q);
                double al = 0.0, be = 0.0, ga = 0.0;
#pragma unroll
                for (int j = 0; j < kRows; ++j) {
                    al = fma(cp[j], cp[j], al);
                    be = fma(cq[j], cq[j], be);
                    ga = fma(cp[j], cq[j], ga);
                }
                al = warp_sum(al);
                be = warp_sum(be);
                ga = warp_sum(ga);
                if (fabs(ga) > 1e-16 * sqrt(al * be) && fabs(ga) > 1e-300) {
                    rotated = true;
                    const double zeta = (be - al) / (2.0 * ga);
                    const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
#pragma unroll
                    for (int j = 0; j < kRows; ++j) {
                        const double vp = cp[j], vq = cq[j];
                        cp[j] = c * vp - s * vq;
                        cq[j] = s * vp + c * vq;
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const double vp = V[k][p], vq = V[k][q];
                        V[k][p] = c * vp - s * vq;
                        V[k][q] = s * vp + c * vq;
                    }
                }
            }
        }
        if (!rotated) break;
    }
    double sv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        double* cc = COL(c);
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < kRows; ++j) acc = fma(cc[j], cc[j], acc);
        sv[c] = sqrt(warp_sum(acc));
    }
#undef COL
    int jmin = 0;
#pragma unroll
    for (int c = 1; c < 4; ++c)
        if (sv[c] < sv[jmin]) jmin = c;

    FitResult res;
    res.fallback = 0;
    double A[4];
    if (sv[jmin] < 1e-12) {  // circle_fitting.cpp:174-175
#pragma unroll
        for (int i = 0; i < 4; ++i) A[i] = V[i][0];
#pragma unroll
        for (int c = 1; c < 4; ++c)
            if (c == jmin) {
#pragma unroll
                for (int i = 0; i < 4; ++i) A[i] = V[i][c];
            }
    } else {
        double Y[4][4], T[4][4], Q[4][4], E[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) acc = fma(V[i][j] * sv[j], V[k][j], acc);
                Y[i][k] = acc;
            }
        // T = H_inv * Y with H_inv = [[0,0,0,.5],[0,1,0,0],[0,0,1,0],[.5,0,0,-2 z_mean]]  (:156-161)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            T[0][k] = 0.5 * Y[3][k];
            T[1][k] = Y[1][k];
            T[2][k] = Y[2][k];
            T[3][k] = 0.5 * Y[0][k] - 2.0 * zm * Y[3][k];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) acc = fma(Y[i][j], T[j][k], acc);
                Q[i][k] = acc;
            }
        // Q = Y H_inv Y is symmetric (Y and H_inv are); symmetrise the rounding noise before Jacobi
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = i + 1; k < 4; ++k) {
                const double m = 0.5 * (Q[i][k] + Q[k][i]);
                Q[i][k] = m;
                Q[k][i] = m;
            }
        jacobi_eig4(Q, E);
        int idx = -1;
        double small = 1000.0;  // :187-197
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (Q[i][i] > 0.0 && Q[i][i] < small) {
                small = Q[i][i];
                idx = i;
            }
        if (idx < 0) {
            // No eigenvalue in (0, 1000): the reference takes eig_gen's index 0 (:187-197).  Q = Y H^-1 Y has exactly
            // one negative eigenvalue (H^-1 has signature (3, 1)), and LAPACK's dgeev - what Armadillo's eig_gen calls -
            // returns it first for this matrix family: 3,000 of 3,000 random large-coordinate clusters with the
            // reference build here (tests/test_gpu_circles.py::test_eigenvalue_fallback_matches_the_reference_build).
            // So the fallback is the eigenvector of the negative eigenvalue.
            res.fallback = 1;
            idx = 0;
            double most_neg = Q[0][0];
#pragma unroll
            for (int i = 1; i < 4; ++i)
                if (Q[i][i] < most_neg) {
                    most_neg = Q[i][i];
                    idx = i;
                }
        }
        double As[4] = {E[0][0], E[1][0], E[2][0], E[3][0]};
#pragma unroll
        for (int c = 1; c < 4; ++c)
            if (c == idx) {
#pragma unroll
                for (int i = 0; i < 4; ++i) As[i] = E[i][c];
            }
        // A = Y^-1 A* = V diag(1/s) V^T A*   (solve(Y, A*), :211)
        double w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) acc = fma(V[i][j], As[i], acc);
            w[j] = acc / sv[j];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double acc = 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) acc = fma(V[i][j], w[j], acc);
            A[i] = acc;
        }
    }
    const double ca = -A[1] / (2.0 * A[0]), cb = -A[2] / (2.0 * A[0]);  // :220-222
    const double r2 = (A[1] * A[1] + A[2] * A[2] - 4.0 * A[0] * A[3]) / (4.0 * A[0] * A[0]);
    res.cx = ca + xm;
    res.cy = cb + ym;
    res.r = sqrt(r2);

    res.mean_angle = mean_angle;
    return res;
}

// centres_only: approxCirclePositions() returns the ACCEPTED centres, and a cluster is accepted only if its mean
// inscribed angle is in range AND its fitted radius is small (:264-271).  The angle statistic does not depend on the
// fit, so it goes first, and a cluster that fails it (every wall segment: a straight run of 50-300 beams whose angle
// is ~pi) skips the SVD fit altogether; what approxCirclePositions() returns is unchanged.  With centres_only = false
// every cluster is fitted (circleRegression() / the per-cluster seams).
template <class Fetch>
__device__ __forceinline__ FitResult warp_circle_fit(Fetch pt, const int n, const int lane, const bool centres_only = false) {
    const double mean_angle = warp_mean_inscribed_angle(pt, n, lane);
    if (centres_only && !angle_in_circle_range(mean_angle)) {  // warp-uniform
        FitResult res;
        res.cx = res.cy = res.r = nan("");
        res.mean_angle = mean_angle;
        res.fallback = 0;
        return res;
    }
    if (n <= 64) return warp_circle_fit_rows<2>(pt, n, lane, mean_angle);   // warp-uniform branch
    if (n <= 128) return warp_circle_fit_rows<4>(pt, n, lane, mean_angle);
    return warp_circle_fit_rows<kRows>(pt, n, lane, mean_angle);
}

__device__ __forceinline__ bool is_circle(const FitResult& f) {
    return f.mean_angle > 1.5708 && f.mean_angle < 2.3562 && f.r < 0.2;  // :264-271
}

struct ScanOut {
    int32_t* n_clusters;  // [B]
    int32_t* segs;        // [B][kMaxClusters][4]
    double* cxr;          // [B][kMaxClusters][4]  cx, cy, r, mean_angle
    uint8_t* flags;       // [B][kMaxClusters]     bit0 = is_circle, bit1 = eigenvalue fallback
    double* xy;           // [B][n_beams][2]       cartesian points (device cos/sin), for the clustering seam
    double* centers;      // [B][max_c][2]
    int32_t* counts;      // [B]
    int centres_only;     // 1: only centers / counts are needed (clusters failing the angle test are not fitted)
};

template <typename T>
__global__ void __launch_bounds__(kCtaThreads, CIRC_MIN_CTAS)
    k_circles_scan(const T* __restrict__ ranges, long long B, int n_beams, int max_c, ScanOut out) {
    __shared__ double r[kMaxBeams];
    __shared__ double2 xy[kMaxBeams];
    __shared__ int keep[kMaxBeams];
    __shared__ Segs seg[kMaxClusters];
    __shared__ double res[kMaxClusters][4];
    __shared__ unsigned char flg[kMaxClusters];
    __shared__ int ncl_s;
    const long long b = blockIdx.x;
    if (b >= B) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double resol = 2 * kPi / (double)n_beams;  // :16
    for (int i = tid; i < n_beams; i += kCtaThreads) {
        const double v = (double)ranges[b * n_beams + i];  // float32 on the wire, widened (landmarks.cpp:65-68)
        r[i] = v;
        double s, c;
        if (i == 0) {
            s = 0.0;  // cos(0.0), sin(0.0)  (:25-26)
            c = 1.0;
        } else {
            sincos(ekf::normalize_angle((double)i * resol), &s, &c);
        }
        xy[i] = make_double2(v * c, v * s);
        if (out.xy && !out.centres_only) {
            out.xy[(b * n_beams + i) * 2] = v * c;
            out.xy[(b * n_beams + i) * 2 + 1] = v * s;
        }
    }
    __syncthreads();
    // runs of consecutive beams with |dr| < 0.2; beam n-1 always opens a new (never flushed) cluster (:30-40)
    for (int i = tid; i < n_beams; i += kCtaThreads) {
        int L = 0;
        if (i <= n_beams - 2) {
            const bool start = (i == 0) || !(fabs(r[i] - r[i - 1]) < kThresh);
            if (start) {
                int e = i + 1;
                while (e <= n_beams - 2 && fabs(r[e] - r[e - 1]) < kThresh) ++e;
                L = e - i;
            }
        }
        keep[i] = (L > 6) ? L : 0;  // :34
    }
    __syncthreads();
    if (warp == 0) {  // ordered compaction of the surviving runs
        int base = 0;
        for (int c0 = 0; c0 < n_beams; c0 += 32) {
            const int i = c0 + lane;
            const int L = (i < n_beams) ? keep[i] : 0;
            const unsigned m = __ballot_sync(0xffffffffu, L > 0);
            if (L > 0) {
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                if (pos < kMaxClusters) seg[pos] = Segs{i, L, 0, 0};
            }
            base += __popc(m);
        }
        if (lane == 0) {
            int ncl = base < kMaxClusters ? base : kMaxClusters;
            if (ncl > 0) {  // wrap merge (:54-70); a single cluster merges with itself and is popped
                const double first = r[seg[0].s1];
                const Segs la = seg[ncl - 1];
                const double last = r[la.s1 + la.l1 - 1];
                if (fabs(first - last) < kThresh) {
                    if (ncl == 1) {
                        ncl = 0;
                    } else {
                        seg[0] = Segs{la.s1, la.l1, seg[0].s1, seg[0].l1};
                        ncl -= 1;
                    }
                }
            }
            ncl_s = ncl;
        }
    }
    __syncthreads();
    const int ncl = ncl_s;
    for (int c = warp; c < ncl; c += kCtaThreads / 32) {
        const Segs sg = seg[c];
        auto fetch = [&](int k) -> double2 { return xy[k < sg.l1 ? sg.s1 + k : sg.s2 + (k - sg.l1)]; };
        const FitResult f = warp_circle_fit(fetch, sg.l1 + sg.l2, lane, out.centres_only != 0);
        if (lane == 0) {
            res[c][0] = f.cx;
            res[c][1] = f.cy;
            res[c][2] = f.r;
            res[c][3] = f.mean_angle;
            flg[c] = (is_circle(f) ? 1 : 0) | (f.fallback ? 2 : 0);
        }
    }
    __syncthreads();
    if (tid == 0) {
        int k = 0;
        for (int c = 0; c < ncl; ++c) {
            if (flg[c] & 1) {
                if (k < max_c && out.centers) {
                    out.centers[(b * max_c + k) * 2] = res[c][0];
                    out.centers[(b * max_c + k) * 2 + 1] = res[c][1];
                }
                ++k;
            }
        }
        if (out.counts) out.counts[b] = k;
        if (out.n_clusters) out.n_clusters[b] = ncl;
    }
    for (int c = tid; c < ncl; c += kCtaThreads) {
        if (out.segs) {
            int32_t* s = out.segs + (b * kMaxClusters + c) * 4;
            s[0] = seg[c].s1;
            s[1] = seg[c].l1;
            s[2] = seg[c].s2;
            s[3] = seg[c].l2;
        }
        if (out.cxr) {
            double* d = out.cxr + (b * kMaxClusters + c) * 4;
            d[0] = res[c][0];
            d[1] = res[c][1];
            d[2] = res[c][2];
            d[3] = res[c][3];
        }
        if (out.flags) out.flags[b * kMaxClusters + c] = flg[c];
    }
}

// circleRegression + classifyCircle on caller-supplied clusters (the set_xy_cluster seam, :96-98)
__global__ void __launch_bounds__(128)
    k_circles_fit_clusters(const double* __restrict__ flat_xy, const int* __restrict__ offsets, int n_clusters,
                           double* __restrict__ cxr, uint8_t* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n_clusters) return;
    const int o = offsets[c], n = offsets[c + 1] - o;
    auto fetch = [&](int k) -> double2 { return make_double2(flat_xy[2 * (o + k)], flat_xy[2 * (o + k) + 1]); };
    const FitResult f = warp_circle_fit(fetch, n, lane);
    if (lane == 0) {
        cxr[4 * c] = f.cx;
        cxr[4 * c + 1] = f.cy;
        cxr[4 * c + 2] = f.r;
        cxr[4 * c + 3] = f.mean_angle;
        flags[c] = (is_circle(f) ? 1 : 0) | (f.fallback ? 2 : 0);
    }
}

}  // namespace circ

struct circles_ctx {
    long long cap = 0;
    int n_beams = 0, device = 0, max_c = 0;
    cudaStream_t stream = nullptr;
    void* d_ranges = nullptr;  // cap * n_beams * 8
    circ::ScanOut o{};
    long long last_B = 0;
    uint64_t launches = 0;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
};

namespace {
template <typename T>
int run_scans(circles_ctx* c, const T* d_ranges, long long B) {
    circ::k_circles_scan<T><<<(unsigned)B, circ::kCtaThreads, 0, c->stream>>>(d_ranges, B, c->n_beams, c->max_c, c->o);
    c->launches += 1;
    c->last_B = B;
    CU(cudaGetLastError());
    return 0;
}
}  // namespace

extern "C" {

const char* circles_last_error(void) { return g_err; }

int circles_create(int64_t max_scans, int n_beams, int max_circles, int device, circles_ctx** out) {
    if (!out) return fail(-1, "null out pointer");
    *out = nullptr;
    if (max_scans <= 0 || n_beams < 2 || max_circles <= 0) return fail(-1, "invalid shape");
    if (n_beams > circ::kMaxBeams) return fail(-2, "n_beams=%d exceeds %d", n_beams, circ::kMaxBeams);
    int rc = check_device(device);
    if (rc) return rc;
    DeviceGuard g(device);
    circles_ctx* c = new (std::nothrow) circles_ctx();
    if (!c) return fail(-3, "out of host memory");
    c->cap = max_scans;
    c->n_beams = n_beams;
    c->device = device;
    c->max_c = max_circles;
    const size_t B = (size_t)max_scans;
    cudaError_t err = cudaSuccess;
    auto A = [&](void** p, size_t bytes) {
        if (err == cudaSuccess) err = cudaMalloc(p, bytes);
    };
    err = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    A(&c->d_ranges, B * n_beams * sizeof(double));
    A((void**)&c->o.n_clusters, B * sizeof(int32_t));
    A((void**)&c->o.segs, B * circ::kMaxClusters * 4 * sizeof(int32_t));
    A((void**)&c->o.cxr, B * circ::kMaxClusters * 4 * sizeof(double));
    A((void**)&c->o.flags, B * circ::kMaxClusters);
    A((void**)&c->o.xy, B * n_beams * 2 * sizeof(double));
    A((void**)&c->o.centers, B * max_circles * 2 * sizeof(double));
    A((void**)&c->o.counts, B * sizeof(int32_t));
    if (err != cudaSuccess) {
        cudaGetLastError();
        int code = fail((int)err, "allocation failed: %s", cudaGetErrorString(err));
        circles_destroy(c);
        return code;
    }
    *out = c;
    return 0;
}

int circles_destroy(circles_ctx* c) {
    if (!c) return 0;
    DeviceGuard g(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    cudaFree(c->d_ranges);
    cudaFree(c->o.n_clusters);
    cudaFree(c->o.segs);
    cudaFree(c->o.cxr);
    cudaFree(c->o.flags);
    cudaFree(c->o.xy);
    cudaFree(c->o.centers);
    cudaFree(c->o.counts);
    if (c->t0) cudaEventDestroy(c->t0);
    if (c->t1) cudaEventDestroy(c->t1);
    if (c->stream) cudaStreamDestroy(c->stream);
    cudaGetLastError();
    delete c;
    return 0;
}

static int fetch_results(circles_ctx* c, long long B, double* centers, int32_t* counts) {
    if (centers)
        CU(cudaMemcpyAsync(centers, c->o.centers, sizeof(double) * 2 * c->max_c * B, cudaMemcpyDeviceToHost, c->stream));
    if (counts) CU(cudaMemcpyAsync(counts, c->o.counts, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int circles_run_f32(circles_ctx* c, const float* ranges, int64_t B, double* centers, int32_t* counts) {
    if (!c || !ranges || B <= 0 || B > c->cap) return fail(-1, "invalid argument");
    DeviceGuard g(c->device);
    CU(cudaMemcpyAsync(c->d_ranges, ranges, sizeof(float) * c->n_beams * B, cudaMemcpyHostToDevice, c->stream));
    int rc = run_scans<float>(c, static_cast<const float*>(c->d_ranges), B);
    if (rc) return rc;
    return fetch_results(c, B, centers, counts);
}

int circles_run_f64(circles_ctx* c, const double* ranges, int64_t B, double* centers, int32_t* counts) {
    if (!c || !ranges || B <= 0 || B > c->cap) return fail(-1, "invalid argument");
    DeviceGuard g(c->device);
    CU(cudaMemcpyAsync(c->d_ranges, ranges, sizeof(double) * c->n_beams * B, cudaMemcpyHostToDevice, c->stream));
    int rc = run_scans<double>(c, static_cast<const double*>(c->d_ranges), B);
    if (rc) return rc;
    return fetch_results(c, B, centers, counts);
}

int circles_run_dev_f32(circles_ctx* c, const float* d_ranges, int64_t B) {
    if (!c || !d_ranges || B <= 0 || B > c->cap) return fail(-1, "invalid argument");
    DeviceGuard g(c->device);
    return run_scans<float>(c, d_ranges, B);
}

int circles_device_outputs(circles_ctx* c, void** d_centers, void** d_counts) {
    if (!c) return fail(-1, "null handle");
    if (d_centers) *d_centers = c->o.centers;
    if (d_counts) *d_counts = c->o.counts;
    return 0;
}

int circles_last_clusters(circles_ctx* c, int64_t scan, int32_t* n_clusters, int32_t* segs, double* cxr,
                          uint8_t* flags, double* xy) {
    if (!c || scan < 0 || scan >= c->last_B) return fail(-1, "invalid argument");
    DeviceGuard g(c->device);
    const int M = circ::kMaxClusters;
    if (n_clusters) CU(cudaMemcpyAsync(n_clusters, c->o.n_clusters + scan, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (segs) CU(cudaMemcpyAsync(segs, c->o.segs + scan * M * 4, sizeof(int32_t) * M * 4, cudaMemcpyDeviceToHost, c->stream));
    if (cxr) CU(cudaMemcpyAsync(cxr, c->o.cxr + scan * M * 4, sizeof(double) * M * 4, cudaMemcpyDeviceToHost, c->stream));
    if (flags) CU(cudaMemcpyAsync(flags, c->o.flags + scan * M, M, cudaMemcpyDeviceToHost, c->stream));
    if (xy) CU(cudaMemcpyAsync(xy, c->o.xy + scan * c->n_beams * 2, sizeof(double) * 2 * c->n_beams, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int circles_max_clusters(void) { return circ::kMaxClusters; }
int circles_max_beams(void) { return circ::kMaxBeams; }

int circles_fit_clusters(circles_ctx* c, const double* flat_xy, const int32_t* sizes, int n_clusters, double* cxr,
                         uint8_t* flags) {
    if (!c || !flat_xy || !sizes || n_clusters <= 0 || !cxr || !flags) return fail(-1, "invalid argument");
    DeviceGuard g(c->device);
    int total = 0;
    int* offs = new (std::nothrow) int[n_clusters + 1];
    if (!offs) return fail(-3, "out of host memory");
    for (int i = 0; i < n_clusters; ++i) {
        if (sizes[i] < 1 || sizes[i] > circ::kMaxBeams) {
            delete[] offs;
            return fail(-2, "cluster %d has %d points (supported: 1..%d)", i, sizes[i], circ::kMaxBeams);
        }
        offs[i] = total;
        total += sizes[i];
    }
    offs[n_clusters] = total;
    double *d_xy = nullptr, *d_cxr = nullptr;
    int* d_off = nullptr;
    uint8_t* d_fl = nullptr;
    cudaError_t e = cudaMalloc(&d_xy, sizeof(double) * 2 * total);
    if (e == cudaSuccess) e = cudaMalloc(&d_off, sizeof(int) * (n_clusters + 1));
    if (e == cudaSuccess) e = cudaMalloc(&d_cxr, sizeof(double) * 4 * n_clusters);
    if (e == cudaSuccess) e = cudaMalloc(&d_fl, n_clusters);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_xy, flat_xy, sizeof(double) * 2 * total, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, offs, sizeof(int) * (n_clusters + 1), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        circ::k_circles_fit_clusters<<<(n_clusters + 3) / 4, 128, 0, c->stream>>>(d_xy, d_off, n_clusters, d_cxr, d_fl);
        c->launches += 1;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(cxr, d_cxr, sizeof(double) * 4 * n_clusters, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(flags, d_fl, n_clusters, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_xy);
    cudaFree(d_off);
    cudaFree(d_cxr);
    cudaFree(d_fl);
    delete[] offs;
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail((int)e, "circles_fit_clusters: %s", cudaGetErrorString(e));
    }
    return 0;
}

int circles_sync(circles_ctx* c) {
    if (!c) return fail(-1, "null handle");
    DeviceGuard g(c->device);
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}
int circles_timer_start(circles_ctx* c) {
    if (!c) return fail(-1, "null handle");
    DeviceGuard g(c->device);
    if (!c->t0) {
        CU(cudaEventCreate(&c->t0));
        CU(cudaEventCreate(&c->t1));
    }
    CU(cudaEventRecord(c->t0, c->stream));
    return 0;
}
int circles_timer_stop(circles_ctx* c, float* ms_out) {
    if (!c || !ms_out || !c->t0) return fail(-1, "timer not started");
    DeviceGuard g(c->device);
    CU(cudaEventRecord(c->t1, c->stream));
    CU(cudaEventSynchronize(c->t1));
    CU(cudaEventElapsedTime(ms_out, c->t0, c->t1));
    return 0;
}
// 1: runs return only what approxCirclePositions() returns (accepted centres + counts); clusters that fail the
// inscribed-angle test are not fitted and circles_last_clusters() reports NaN for them.  0 (default): every cluster is
// fitted, as circleRegression() does.  The accepted centres are identical in both modes.
int circles_set_centres_only(circles_ctx* c, int on) {
    if (!c) return fail(-1, "null handle");
    c->o.centres_only = on ? 1 : 0;
    return 0;
}

int circles_launch_count(circles_ctx* c, uint64_t* out) {
    if (!c || !out) return fail(-1, "null argument");
    *out = c->launches;
    return 0;
}

}  // extern "C"
