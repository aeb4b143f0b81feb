// Consistency read-out of a batch of filters (no reference counterpart: the reference keeps one filter and never
// scores its covariance).  For every filter b of an ekf_batch, in any of its three Sigma layouts:
//   marginals : P = Sigma[0:3, 0:3] (pose, state order theta, x, y) and the 2 x 2 block L_i of every landmark slot;
//   NEES      : e^T P^-1 e of the pose (3 x 3 Cholesky) and of every scored landmark slot (closed-form 2 x 2 inverse)
//               against caller-supplied truth;
//   partials  : {sum NEES_pose, sum NEES_pose^2, #pose, sum NEES_lm, sum NEES_lm^2, #lm, #singular pose, #singular lm}
//               over the batch, reduced in a fixed order (per lane in filter order, warp shuffle tree, warps of a CTA in
//               index order, CTAs in index order by the last CTA to finish), so two calls on the same state and device
//               return bit-identical partials.  No floating-point atomics.
// Only stored entries (r <= c) are read, through the layouts' own index helpers, so every value is bit-identical to
// entry (r, c) of ekf_batch_get_sigma().  The kernel reads Sigma, the state, the init flags and the known lists and
// writes nothing the filters own.
// k_batch_nis reads out the NIS accumulators the step kernels' NIS variants keep (ekf_batch_set_nis), with the same
// fixed-order reduction (reduce_batch_partials).
#pragma once
#include "ekf_fused_sym.cuh"
#include "ekf_fused_tile.cuh"

namespace ekf {

// Sigma(r, c), r <= c, of filter b in each batch layout
struct TileAt {  // n = 20: register-fragment tile layout (ekf_fused_tile.cuh)
    const double* sigma;
    __device__ double operator()(long long b, int r, int c) const { return sigma[b * tile::kStride + tile::tile_at(r, c)]; }
};
struct StairAt {  // n <= 64, n != 20: symmetric block staircase (ekf_fused_sym.cuh)
    const double* sigma;
    long long stride;
    int N;
    __device__ double operator()(long long b, int r, int c) const { return sigma[b * stride + stair_at(r, c, N)]; }
};
struct WideAt {  // 64 < n <= 1,024: dense N x ld rows, upper triangle (ekf_batch_wide.cuh)
    const double* sigma;
    long long stride, ld;
    __device__ double operator()(long long b, int r, int c) const { return sigma[b * stride + r * ld + c]; }
};

constexpr int kConsWarps = 8;  // warps per CTA of k_batch_consistency and k_batch_nis

// Batch total of K per-lane partials in a fixed order: warp (shuffle tree), then the kConsWarps warps of the CTA in index
// order into partials[blockIdx.x][K], then CTAs in index order by the last CTA to finish, into out[K].  `done` counts
// finished CTAs and is zero between launches (the last CTA resets it).  Every thread of the CTA calls this, with
// lane = threadIdx.x % 32 and warp = threadIdx.x / 32.
template <int K>
__device__ __forceinline__ void reduce_batch_partials(const double (&acc)[K], const int lane, const int warp,
                                                      double* partials, unsigned int* done, double* out) {
    __shared__ double red[kConsWarps][K];
    __shared__ bool last;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double v = acc[k];
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (int w = 0; w < kConsWarps; ++w) s += red[w][threadIdx.x];
        partials[K * blockIdx.x + threadIdx.x] = s;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (unsigned g = 0; g < gridDim.x; ++g) s += __ldcg(partials + K * g + threadIdx.x);
        out[threadIdx.x] = s;
    }
    if (threadIdx.x == 0) *done = 0;
}

struct ConsistencyParams {
    const double* state;       // [B][st_stride]: theta, x, y, m1x, m1y, ...
    const int32_t* init_flag;  // [B]
    const uint8_t* known;      // [B][n]
    const double* truth;       // [B][3] = {x, y, theta}; null: marginals only
    const double* lm_truth;    // [n][2] (lm_stride 0) or [B][n][2] (lm_stride 2n); NaN = not scored; null = no landmarks
    double* per_filter;        // [B][3] = {NEES_pose, sum_i NEES_i, count_i}, optional
    double* pose_cov;          // [B][6] = 00, 01, 02, 11, 12, 22, optional
    double* lm_cov;            // [B][n][3] = xx, xy, yy, optional
    double* partials;          // [gridDim.x][8]
    unsigned int* done;        // CTAs finished; zero between launches (the last CTA resets it)
    double* out8;              // batch partial, written by the last CTA
    long long B, st_stride, lm_stride;
    int n;
};

template <class At>
__global__ void __launch_bounds__(kConsWarps * 32) k_batch_consistency(ConsistencyParams p, At at) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // this lane's share of the batch partial
    for (long long b = (long long)blockIdx.x * kConsWarps + warp; b < p.B; b += (long long)gridDim.x * kConsWarps) {
        const double* st = p.state + b * p.st_stride;
        double pose_nees = nan;
        if (lane == 0) {
            const double a00 = at(b, 0, 0), a01 = at(b, 0, 1), a02 = at(b, 0, 2);
            const double a11 = at(b, 1, 1), a12 = at(b, 1, 2), a22 = at(b, 2, 2);
            if (p.pose_cov) {
                double* o = p.pose_cov + 6 * b;
                o[0] = a00, o[1] = a01, o[2] = a02, o[3] = a11, o[4] = a12, o[5] = a22;
            }
            if (p.truth) {
                const double* t = p.truth + 3 * b;
                const double e0 = normalize_angle(st[0] - t[2]), e1 = st[1] - t[0], e2 = st[2] - t[1];
                // P = L L^T; a pivot that is not positive and finite makes the block singular
                const double d0 = a00;
                const double l00 = sqrt(d0), l10 = a01 / l00, l20 = a02 / l00;
                const double d1 = a11 - l10 * l10;
                const double l11 = sqrt(d1), l21 = (a12 - l20 * l10) / l11;
                const double d2 = a22 - l20 * l20 - l21 * l21;
                const bool pd = d0 > 0.0 && d1 > 0.0 && d2 > 0.0 && isfinite(d0) && isfinite(d1) && isfinite(d2);
                if (!pd) {
                    acc[6] += 1.0;
                } else if (isfinite(e0) && isfinite(e1) && isfinite(e2)) {
                    const double y0 = e0 / l00, y1 = (e1 - l10 * y0) / l11, y2 = (e2 - l20 * y0 - l21 * y1) / sqrt(d2);
                    pose_nees = y0 * y0 + y1 * y1 + y2 * y2;
                    acc[0] += pose_nees;
                    acc[1] += pose_nees * pose_nees;
                    acc[2] += 1.0;
                }
            }
        }
        const bool all_slots = p.init_flag[b] != 0;
        double lm_sum = 0.0, lm_cnt = 0.0;
        for (int i = lane; i < p.n; i += 32) {
            const int r = 3 + 2 * i;
            const double a = at(b, r, r), c = at(b, r, r + 1), d = at(b, r + 1, r + 1);
            if (p.lm_cov) {
                double* o = p.lm_cov + 3 * (b * p.n + i);
                o[0] = a, o[1] = c, o[2] = d;
            }
            if (!p.truth || !p.lm_truth || !(all_slots || p.known[b * p.n + i])) continue;
            const double* t = p.lm_truth + b * p.lm_stride + 2 * i;
            if (!isfinite(t[0]) || !isfinite(t[1])) continue;
            const double ex = st[r] - t[0], ey = st[r + 1] - t[1];
            const double det = a * d - c * c;
            if (!(a > 0.0 && det > 0.0 && isfinite(det))) {
                acc[7] += 1.0;
                continue;
            }
            const double v = (d * ex * ex - 2.0 * c * ex * ey + a * ey * ey) / det;
            lm_sum += v;
            lm_cnt += 1.0;
            acc[3] += v;
            acc[4] += v * v;
            acc[5] += 1.0;
        }
        if (p.per_filter) {
            for (int off = 16; off > 0; off >>= 1) {
                lm_sum += __shfl_xor_sync(0xffffffffu, lm_sum, off);
                lm_cnt += __shfl_xor_sync(0xffffffffu, lm_cnt, off);
            }
            if (lane == 0) {
                double* o = p.per_filter + 3 * b;
                o[0] = pose_nees, o[1] = lm_sum, o[2] = lm_cnt;
            }
        }
    }
    if (!p.out8) return;
    reduce_batch_partials<8>(acc, lane, warp, p.partials, p.done, p.out8);
}

// NIS read-out of a batch (ekf_batch_nis): the [B][4] accumulators {sum NIS, sum NIS^2, #scored, #non-finite} that
// the step kernels' NIS variants keep, copied to per_filter (optional) and summed over the batch in the fixed order of
// reduce_batch_partials: each thread adds its filters b = thread, thread + threads, ... in filter order first.  reset
// zeroes the accumulators after they were read (each filter is read and cleared by the same thread).
__global__ void __launch_bounds__(kConsWarps * 32) k_batch_nis(double* acc4, long long B, double* per_filter,
                                                               int reset, double* partials, unsigned int* done,
                                                               double* out4) {
    double acc[4] = {0, 0, 0, 0};
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        double v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[k] = acc4[4 * b + k];
            acc[k] += v[k];
        }
        if (per_filter)
#pragma unroll
            for (int k = 0; k < 4; ++k) per_filter[4 * b + k] = v[k];
        if (reset)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc4[4 * b + k] = 0.0;
    }
    reduce_batch_partials<4>(acc, threadIdx.x & 31, threadIdx.x >> 5, partials, done, out4);
}

}  // namespace ekf
