// Engine 2: one filter whose covariance lives in HBM (maps too large for shared memory; cfg4 has
// n = 8,192 landmarks, Sigma = 16,387^2 fp64 = 2.1 GB).  Sigma is row-major with the row stride `ld`
// padded to a multiple of 16 doubles (128 B) so that every row starts on a cache line and 256-bit
// loads/stores are aligned.  Per landmark correction the work is
//   gain  : O(N)  — 5 rows + 5 columns of Sigma -> W = Hj Sigma (2 x N), K = Sigma Hj^T S^-1 (N x 2), state
//   sweep : O(N^2)— Sigma -= sum K W, streamed once through the SMs: one HBM read + one HBM write of Sigma
// (both kernels live in ekf_large_delayed.cuh; this header holds prediction, association and shared pieces).
// Restates rigid2d/src/ekf_slam.cpp:55-106, :108-197, :200-214, :217-276, :278-402.
#pragma once
#include "ekf_math.cuh"

namespace ekf {

// What the association step decided for one measurement; consumed by gain + sweep without a host round trip.
struct UpdateCmd {
    int do_update;  // 1: correct landmark `lm` with (sx, sy)
    int lm;
    int created;    // a new landmark was initialised for this measurement
    int pad;
    double sx, sy;
};

struct AssocPartial {
    double best, second;
    int best_i;
    int pad;
};

// Programmatic dependent launch (PDL): the streamed engine's short kernels form a serial chain on one stream, and a
// correction is ~9 us of which a good part is launch latency.  A kernel launched with the programmatic-stream-
// serialization attribute may be scheduled while its predecessor still runs; it must not touch the predecessor's
// results before griddepcontrol.wait (which returns once the predecessor has completed and flushed).  Triggering the
// dependents at entry is always safe for that reason.  Without the launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_prologue() {
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---------------------------------------------------------------- prediction (ekf_slam.cpp:55-106)
// One warp: lane 0 does the motion model, state[0..2], the 3x3 robot block of At*Sigma*At^T + Q, and (a1, a2) for the
// strips; lane j < pending carries pending factor j across the prediction (ekf_large_delayed.cuh).  The row-sharded
// engine runs it on every rank: `sig` is then the rank's 3 x ld copy of rows 0..2, or its own rows on rank 0.
__global__ void k_large_motion(double* __restrict__ state, double* __restrict__ sig, long long ld, double dtheta,
                               double dx, double* __restrict__ motion_out, double2* __restrict__ Kp,
                               double2* __restrict__ Wp, int pending) {
    pdl_prologue();
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    Motion m = {};
    if (threadIdx.x == 0) m = motion_model(state[0], dtheta, dx);
    const double a1 = __shfl_sync(0xffffffffu, m.a1, 0), a2 = __shfl_sync(0xffffffffu, m.a2, 0);
    {
        const int j = threadIdx.x;
        if (j < pending) {  // K_j[1] += a1 K_j[0], K_j[2] += a2 K_j[0]; likewise the columns 1, 2 of W_j
            double2* K = Kp + (long long)j * ld;
            double2* W = Wp + (long long)j * ld;
            const double2 k0 = K[0], w0 = W[0];
            K[1] = make_double2(fma(a1, k0.x, K[1].x), fma(a1, k0.y, K[1].y));
            K[2] = make_double2(fma(a2, k0.x, K[2].x), fma(a2, k0.y, K[2].y));
            W[1] = make_double2(fma(a1, w0.x, W[1].x), fma(a1, w0.y, W[1].y));
            W[2] = make_double2(fma(a2, w0.x, W[2].x), fma(a2, w0.y, W[2].y));
        }
    }
    if (threadIdx.x != 0) return;
    double s[3][3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) s[r][c] = sig[r * ld + c];
    for (int c = 0; c < 3; ++c) {
        s[1][c] = fma(m.a1, s[0][c], s[1][c]);
        s[2][c] = fma(m.a2, s[0][c], s[2][c]);
    }
    for (int r = 0; r < 3; ++r) {
        s[r][1] = fma(s[r][0], m.a1, s[r][1]);
        s[r][2] = fma(s[r][0], m.a2, s[r][2]);
    }
    s[0][0] += kQ;
    s[1][1] += kQ;
    s[2][2] += kQ;
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) sig[r * ld + c] = s[r][c];
    state[0] = state[0] + m.u0;
    state[1] = state[1] + m.u1;
    state[2] = state[2] + m.u2;
    motion_out[0] = m.a1;
    motion_out[1] = m.a2;
}

// Robot-landmark strips: rows 1,2 += a*row0 and cols 1,2 += a*col0 for indices k >= 3.  6N doubles touched.
__global__ void k_large_predict_strips(double* __restrict__ sig, long long ld, int N,
                                       const double* __restrict__ motion) {
    pdl_prologue();
    const int k = 3 + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    const double a1 = motion[0], a2 = motion[1];
    const double r0 = sig[k];
    sig[ld + k] = fma(a1, r0, sig[ld + k]);
    sig[2 * ld + k] = fma(a2, r0, sig[2 * ld + k]);
    double* row = sig + (long long)k * ld;
    const double c0 = row[0];
    row[1] = fma(c0, a1, row[1]);
    row[2] = fma(c0, a2, row[2]);
}

// First measurement() call: every slot initialised from its reading (ekf_slam.cpp:113-128).  Also snapshots
// the entry-time pose, which measurement() keeps using for every landmark of the call (:109-111).
__global__ void k_large_init_landmarks(double* __restrict__ state, const double* __restrict__ xy, int n,
                                       int32_t* __restrict__ init_flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *init_flag = 1;
    if (i >= n) return;
    double mx, my;
    landmark_from_reading(xy[2 * i], xy[2 * i + 1], state[0], state[1], state[2], mx, my);
    state[3 + 2 * i] = mx;
    state[4 + 2 * i] = my;
}

// ---------------------------------------------------------------- association (ekf_slam.cpp:217-276, 291-330)
// Mahalanobis distance of measurement j to every known landmark in parallel, block argmin with lowest-index
// tie-break, then the last block to finish reduces the per-block partials and takes the decision
// (new landmark / update / drop) on the device.
__device__ __forceinline__ void assoc_merge(double& best, double& second, int& best_i, double ob, double os, int oi) {
    if (better(ob, oi, best, best_i)) {
        second = fmin(best, os);
        best = ob;
        best_i = oi;
    } else {
        second = fmin(second, fmin(ob, os));
    }
}

// Distances to the landmarks [i_begin, i_end), grid-strided, then the minimum and runner-up over the grid: warp
// shuffles, the CTA's warps, and the last CTA to finish merges the per-CTA partials in CTA order.  Returns true on
// thread 0 of that last CTA only, with the grid's result in best / second / best_i.  Rows 0..2 of Sigma are read from
// `robot`, rows 3+2i and 4+2i from `lm_rows`, which holds the global rows from r0 on.
__device__ __forceinline__ bool assoc_scan(const double* __restrict__ robot, const double* __restrict__ lm_rows,
                                           long long ld, long long r0, int i_begin, int i_end,
                                           const double* __restrict__ state, double zr, double zphi, double theta,
                                           double x, double y, AssocPartial* __restrict__ partials,
                                           unsigned int* __restrict__ done_counter, double& best, double& second,
                                           int& best_i) {
    __shared__ AssocPartial sh[8];
    __shared__ bool is_last;
    best = INFINITY;
    second = INFINITY;
    best_i = 0x7fffffff;
    for (int i = i_begin + blockIdx.x * blockDim.x + threadIdx.x; i < i_end; i += gridDim.x * blockDim.x) {
        const double* lm = lm_rows + ((3 + 2 * (long long)i) - r0) * ld;
        double d = maha_distance_rows(robot, lm, ld, i, state[3 + 2 * i], state[4 + 2 * i], zr, zphi, theta, x, y);
        if (!(d == d)) d = INFINITY;
        if (d < best) {
            second = best;
            best = d;
            best_i = i;
        } else if (d < second) {
            second = d;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, off);
        const double os = __shfl_xor_sync(0xffffffffu, second, off);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, off);
        assoc_merge(best, second, best_i, ob, os, oi);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) sh[warp] = AssocPartial{best, second, best_i, 0};
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) assoc_merge(best, second, best_i, sh[w].best, sh[w].second, sh[w].best_i);
        partials[blockIdx.x] = AssocPartial{best, second, best_i, 0};
        __threadfence();
        const unsigned int t = atomicAdd(done_counter, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last || threadIdx.x != 0) return false;
    __threadfence();
    best = INFINITY;
    second = INFINITY;
    best_i = 0x7fffffff;
    for (unsigned int b = 0; b < gridDim.x; ++b) {
        const volatile AssocPartial* pp = partials + b;
        assoc_merge(best, second, best_i, pp->best, pp->second, pp->best_i);
    }
    *done_counter = 0;  // re-arm for the next measurement (stream-ordered)
    return true;
}

// The decision for measurement j = (sx, sy) from the merged minimum (ekf_slam.cpp:293-330): a new landmark when no
// known one is within kGateNew, an update when the distance is below kGateUpdate.  Writes the command block, the
// new landmark's state and known count, and those of the four outputs that are not null.
__device__ __forceinline__ void assoc_decide(double best, double second, int best_i, int known_count, int n, int j,
                                             double sx, double sy, double theta, double x, double y,
                                             double* __restrict__ state, int* __restrict__ known_count_p,
                                             UpdateCmd* __restrict__ cmd, int32_t* __restrict__ assoc_out,
                                             double* __restrict__ dmin_out, double* __restrict__ second_out,
                                             uint8_t* __restrict__ created_out) {
    double min_d = kGateNew;
    int min_idx = known_count;
    if (best < kGateNew) {
        min_d = best;
        min_idx = best_i;
        second = fmin(second, kGateNew);
    } else {
        second = best;
    }
    if (dmin_out) dmin_out[j] = min_d;
    if (second_out) second_out[j] = second;
    int created = 0;
    if (min_idx == known_count && min_idx < n) {  // ekf_slam.cpp:318-327
        double mx, my;
        landmark_from_reading(sx, sy, theta, x, y, mx, my);
        state[3 + 2 * min_idx] = mx;
        state[4 + 2 * min_idx] = my;
        *known_count_p = known_count + 1;
        min_d = 0.0;
        created = 1;
    }
    const int upd = min_d < kGateUpdate;  // :330
    cmd->do_update = upd;
    cmd->lm = min_idx;
    cmd->created = created;
    cmd->sx = sx;
    cmd->sy = sy;
    if (assoc_out) assoc_out[j] = upd ? min_idx : -1;
    if (created_out) created_out[j] = (uint8_t)created;
}

__global__ void __launch_bounds__(256)
    k_large_assoc(const double* __restrict__ sig, long long ld, double* __restrict__ state, int n,
                  const double* __restrict__ meas, int j, int* __restrict__ known_count_p,
                  AssocPartial* __restrict__ partials, unsigned int* __restrict__ done_counter,
                  UpdateCmd* __restrict__ cmd, int32_t* __restrict__ assoc_out, double* __restrict__ dmin_out,
                  double* __restrict__ second_out, uint8_t* __restrict__ created_out) {
    const int known_count = *known_count_p;
    const double sx = meas[2 * j], sy = meas[2 * j + 1];
    double zr, zphi;
    range_bearing(sx, sy, zr, zphi);
    const double theta = state[0], x = state[1], y = state[2];
    double best, second;
    int best_i;
    if (!assoc_scan(sig, sig, ld, 0, 0, known_count, state, zr, zphi, theta, x, y, partials, done_counter, best,
                    second, best_i))
        return;
    assoc_decide(best, second, best_i, known_count, n, j, sx, sy, theta, x, y, state, known_count_p, cmd, assoc_out,
                 dmin_out, second_out, created_out);
}

// ---------------------------------------------------------------- 256-bit global accesses (LDG/STG.E.256 on sm_100a)
__device__ __forceinline__ void ld256(const double* p, double& a, double& b, double& c, double& d) {
    asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void st256(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

}  // namespace ekf
