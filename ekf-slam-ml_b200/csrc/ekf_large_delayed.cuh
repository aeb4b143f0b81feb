// Delayed application of the rank-2 covariance updates of the streamed engine.
//
// The reference applies Sigma <- Sigma - K W after every landmark correction (ekf_slam.cpp:191-192); for a large
// map that is one full HBM read + write of Sigma per correction.  Here up to kMaxPending corrections are kept as
// factor pairs (K_j, W_j) and applied in ONE sweep:  Sigma <- Sigma - sum_j K_j W_j.  The next correction only needs
// five rows of the CURRENT covariance; they are rebuilt on the fly from Sigma_0 and the pending factors.  Every element goes through exactly the same sequence of FMAs as with sequential sweeps
// (v = fma(-k.y, w.y, fma(-k.x, w.x, v)) for j = 0, 1, ...), so the result is bit-identical — only the HBM traffic
// changes: 16 N^2 bytes per SWEEP instead of per correction.
#pragma once
#include "ekf_large.cuh"

namespace ekf {

// Capacity (factor slots) and default depth of the delayed application.  Up to 14 pending corrections the sweep is
// still a copy (0.90 of the measured HBM peak at N = 16,387: the DMMA time hides behind it) - that is the default.
// Deeper groups (15..20, ekf_set_max_pending) go through the 256-column tiles of k_large_sweep_mma: fewer passes over
// Sigma per correction and more corrections/s (cfg4: 18.6k against 16.5k at 20), but the sweep is then bound by the
// FP64 pipe, not by HBM (0.66 of the copy peak per sweep period).
#ifndef EKF_MAX_PENDING
#define EKF_MAX_PENDING 20
#endif
constexpr int kMaxPending = EKF_MAX_PENDING;
constexpr int kDefaultPending = kMaxPending < 14 ? kMaxPending : 14;

struct GainSharedP {
    Hj h;
    Sym2 si;
    double nu0, nu1;
    double2 Kidx[kMaxPending][5];  // K_j[idx_a], a = 0..4
};

__device__ __forceinline__ double apply_factor(double v, double2 k, double2 w) {
    return fma(-k.y, w.y, fma(-k.x, w.x, v));
}

// ---------------------------------------------------------------- gain arithmetic shared by the streamed engine's
// k_large_gain_p and the wide batch engine (ekf_batch_wide.cuh): both run exactly these expressions, so a filter of a
// wide batch is bit-identical to a streamed filter.  `g.Kidx[j][a]` holds K_j at the five indices {0, 1, 2, i3, i4}.

// Lane `lane` of the scalar warp owns entry (a, l) of the 5 x 5 block {0, 1, 2, i3, i3 + 1}^2 (lanes 25..31 repeat (0, 0)).
struct GainBlockEntry {
    int a, l;
    long long ida, idl;
};
__device__ __forceinline__ GainBlockEntry gain_block_entry(int lane, int i3) {
    GainBlockEntry e;
    e.a = lane < 25 ? lane / 5 : 0;
    e.l = lane < 25 ? lane - 5 * (lane / 5) : 0;
    e.ida = e.a < 3 ? e.a : i3 + (e.a - 3);
    e.idl = e.l < 3 ? e.l : i3 + (e.l - 3);
    return e;
}

// S^-1 and the innovation nu = z - h(x) from H_j, W = H_j Sigma at the five columns {0, 1, 2, i3, i4} and the measured
// range and bearing.  Also used by the row-sharded engine (sharded/sharded.cu).
__device__ __forceinline__ void gain_scalars(const Hj& h, const double2 (&w5)[5], double sx, double sy, const Noise& nz,
                                             Sym2& si, double& nu0, double& nu1) {
    const double s00 = h_row0(h, w5[1].x, w5[2].x, w5[3].x, w5[4].x) + nz.r0;
    const double s01 = h_row1(h, w5[0].x, w5[1].x, w5[2].x, w5[3].x, w5[4].x);
    const double s10 = h_row0(h, w5[1].y, w5[2].y, w5[3].y, w5[4].y);
    const double s11 = h_row1(h, w5[0].y, w5[1].y, w5[2].y, w5[3].y, w5[4].y) + nz.r1;
    si = inv2x2(s00, s01, s10, s11);
    double zr, zphi;
    range_bearing(sx, sy, zr, zphi);
    nu0 = __dsub_rn(zr, h.zr);
    nu1 = normalize_angle(__dsub_rn(zphi, h.zphi));
}

// K[k] = W[:, k]^T S^-1 and the corrected state entry k (returned) from W[:, k] = w and the state entry st_k.
__device__ __forceinline__ double gain_state(const Sym2& si, const double& nu0, const double& nu1, double2 w, double st_k, long long k,
                                             double2& k_out) {
    const double k0 = fma(w.y, si.i10, w.x * si.i00);
    const double k1 = fma(w.y, si.i11, w.x * si.i01);
    k_out = make_double2(k0, k1);
    double ns = st_k + fma(k1, nu1, k0 * nu0);
    if (k == 0) ns = normalize_angle(ns);  // ekf_slam.cpp:187
    return ns;
}

// One full warp: `v` = Sigma_0(id_a, id_l) of the lane's entry.  Rebuilds the current block with the p pending factors,
// then lane 0 leaves H_j, S^-1 and the innovation in g.
__device__ __forceinline__ void gain_block(int lane, const GainBlockEntry& e, double v, const double2* Wp, long long ld,
                                           int p, const Hj& h, double sx, double sy, const Noise& nz, GainSharedP& g) {
#pragma unroll 4
    for (int j = 0; j < p; ++j) v = apply_factor(v, g.Kidx[j][e.a], Wp[(long long)j * ld + e.idl]);
    // column l of the block: s[a'] = Sigma(id_a', id_l) sits in lane 5 a' + l
    const int l = e.l;
    const double s0 = __shfl_sync(0xffffffffu, v, l), s1 = __shfl_sync(0xffffffffu, v, 5 + l),
                 s2 = __shfl_sync(0xffffffffu, v, 10 + l), s3 = __shfl_sync(0xffffffffu, v, 15 + l),
                 s4 = __shfl_sync(0xffffffffu, v, 20 + l);
    const double w0 = h_row0(h, s1, s2, s3, s4), w1 = h_row1(h, s0, s1, s2, s3, s4);  // W[:, id_l]
    double2 w5[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) {  // lanes 0..4 hold columns 0..4
        w5[c].x = __shfl_sync(0xffffffffu, w0, c);
        w5[c].y = __shfl_sync(0xffffffffu, w1, c);
    }
    if (lane == 0) {
        g.h = h;
        gain_scalars(h, w5, sx, sy, nz, g.si, g.nu0, g.nu1);
    }
}

// Column k of the five rows {0, 1, 2, i3, i4}: Sigma_0 entries in s0..s4 on entry, current entries on return.
__device__ __forceinline__ void gain_rows_rebuild(double& s0, double& s1, double& s2, double& s3, double& s4,
                                                  const double2* Wp, long long ld, long long k, int p,
                                                  const GainSharedP& g) {
#pragma unroll 4
    for (int j = 0; j < p; ++j) {
        const double2 wj = Wp[(long long)j * ld + k];  // W_j[:, k]
        s0 = apply_factor(s0, g.Kidx[j][0], wj);
        s1 = apply_factor(s1, g.Kidx[j][1], wj);
        s2 = apply_factor(s2, g.Kidx[j][2], wj);
        s3 = apply_factor(s3, g.Kidx[j][3], wj);
        s4 = apply_factor(s4, g.Kidx[j][4], wj);
    }
}

// W_j[:, k], K_j[k] and the corrected state entry k (returned) from the current rows s0..s4 and state entry st_k.
__device__ __forceinline__ double gain_column(const GainSharedP& g, double s0, double s1, double s2, double s3,
                                              double s4, double st_k, long long k, double2& w_out, double2& k_out) {
    const Hj h = g.h;
    const double2 w = make_double2(h_row0(h, s1, s2, s3, s4), h_row1(h, s0, s1, s2, s3, s4));
    w_out = w;
    return gain_state(g.si, g.nu0, g.nu1, w, st_k, k, k_out);
}

// Correction number `p` of the current group: writes (K_p, W_p), reads Sigma_0 and the factors j < p.
// state_in is never written (the new state goes to state_out), so no CTA can observe a half-updated state.
//
// W = Hj Sigma comes from the five ROWS {0, 1, 2, 3+2i, 4+2i} of the current covariance (coalesced), rebuilt from
// Sigma_0 and the pending factors; K = Sigma Hj^T S^-1 is formed as W^T S^-1 (ekf_slam.cpp:178 with Sigma = Sigma^T,
// which the reference's (I - K H) Sigma keeps to rounding, SURVEY.md §8e) so no strided column of Sigma is touched.
//
// CTA = 8 column warps + 1 scalar warp (kGainThreads = 288).  The scalar warp fetches the pending K pairs at the
// five indices, releases the column warps (named barrier 1), and then does the O(1) part - S from the 5 x 5 block
// with one block entry per lane, its inverse, the innovation with its two atan2 - while the column warps are
// already streaming their five row entries and the pending W pairs; they meet again at named barrier 2.  The
// scalar chain (~2.5 us of dependent latency) used to sit in front of everything.
constexpr int kGainThreads = 288;
__device__ __forceinline__ void named_bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// NIS variants (the single filter's ekf_set_nis): nis_flags bits of the gain kernel.
enum : int {
    kNisScore = 1,  // measurement(): the correction is scored (the filter's landmarks were initialised before the call)
    kNisFold = 2,   // first gain of a call: fold the previous call's sums into the accumulators before scoring
};
// acc = {sum, sum^2, #scored, #non-finite} accumulators, then the sums of the open call: the first gain of a call adds
// the previous call's sums to the accumulators and zeroes them, each scored correction adds its NIS to them, so every
// call is summed on its own, in correction order, and added as a whole (the rule of the batch kernels).
__device__ __forceinline__ void gain_nis(const GainSharedP& g, const UpdateCmd* __restrict__ cmd, bool active,
                                         double* __restrict__ acc, double* __restrict__ nis_out, int nis_flags) {
    if (nis_flags & kNisFold) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            acc[k] += acc[4 + k];
            acc[4 + k] = 0.0;
        }
    }
    // data_association(): every applied correction except that of a landmark the same reading created
    const bool score = cmd ? (cmd->do_update && !cmd->created) : (nis_flags & kNisScore) != 0;
    if (active && score) {
        const double v = nis(g.si, g.nu0, g.nu1);
        *nis_out = v;
        nis_add(acc + 4, v);
    }
}

// k_large_gain_p<NIS, NOISE> runs it with R from `nz` (the single filter's row, ekf_set_noise) under NOISE, otherwise
// with the reference's.  NIS (ekf_set_nis): lane 0 of the scalar warp in CTA 0 scores the correction (gain_nis) into
// nis_acc (the handle's 8 accumulators) and writes its value to *nis_out (the call's slot of this correction).
template <bool NIS>
__device__ __forceinline__ void large_gain_p(const double* __restrict__ sig, long long ld, int N,
                                             const double* __restrict__ state_in, double* __restrict__ state_out,
                                             const double* __restrict__ pose_src, const UpdateCmd* __restrict__ cmd,
                                             int lm_arg, double sx_arg, double sy_arg, double2* __restrict__ Kp,
                                             double2* __restrict__ Wp, int p, const Noise& nz, double* nis_acc,
                                             double* nis_out, int nis_flags) {
    __shared__ GainSharedP g;
    pdl_prologue();
    int lm = lm_arg;
    double sx = sx_arg, sy = sy_arg;
    int active = 1;
    if (cmd) {  // every thread reads the (tiny, uniform) command block itself
        active = cmd->do_update;
        lm = cmd->lm;
        sx = cmd->sx;
        sy = cmd->sy;
    }
    const int i3 = 3 + 2 * lm, i4 = i3 + 1;
    if (threadIdx.x >= 256) {
        // ------------------------------------------------------------ scalar warp
        const int lane = threadIdx.x - 256;
        if (active) {
            if (lane < 5) {
                const long long ida = lane < 3 ? lane : i3 + (lane - 3);
                for (int j = 0; j < p; ++j) g.Kidx[j][lane] = Kp[(long long)j * ld + ida];
            }
        }
        __syncwarp();
        named_bar_sync(1, kGainThreads);
        if (active) {
            const GainBlockEntry e = gain_block_entry(lane, i3);
            const Hj h = make_hj(state_in[i3], state_in[i3 + 1], pose_src[0], pose_src[1], pose_src[2]);
            gain_block(lane, e, sig[e.ida * ld + e.idl], Wp, ld, p, h, sx, sy, nz, g);
        }
        if (NIS && lane == 0 && blockIdx.x == 0) gain_nis(g, cmd, active, nis_acc, nis_out, nis_flags);
        __syncwarp();
        named_bar_sync(2, kGainThreads);
        return;
    }
    // ---------------------------------------------------------------- column warps
    const long long k = (long long)blockIdx.x * 256 + threadIdx.x;
    const bool in_range = k < ld, live = in_range && k < N && active;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0, st_k = 0.0;
    if (live) {  // in flight while the scalar warp fetches the K pairs
        s0 = sig[k], s1 = sig[ld + k], s2 = sig[2 * ld + k], s3 = sig[i3 * ld + k], s4 = sig[i4 * ld + k];
        st_k = state_in[k];
    }
    named_bar_sync(1, kGainThreads);
    if (live) gain_rows_rebuild(s0, s1, s2, s3, s4, Wp, ld, k, p, g);
    named_bar_sync(2, kGainThreads);
    if (!in_range) return;
    double2* Kout = Kp + (long long)p * ld;
    double2* Wout = Wp + (long long)p * ld;
    if (!live) {  // padding entries and dropped measurements contribute a zero factor
        Kout[k] = make_double2(0.0, 0.0);
        Wout[k] = make_double2(0.0, 0.0);
        if (k < N) state_out[k] = state_in[k];
        return;
    }
    double2 wk, kk;
    state_out[k] = gain_column(g, s0, s1, s2, s3, s4, st_k, k, wk, kk);
    Wout[k] = wk;
    Kout[k] = kk;
}
template <bool NIS, bool NOISE>
__global__ void __launch_bounds__(kGainThreads)
    k_large_gain_p(const double* __restrict__ sig, long long ld, int N, const double* __restrict__ state_in,
                   double* __restrict__ state_out, const double* __restrict__ pose_src, const UpdateCmd* __restrict__ cmd,
                   int lm_arg, double sx_arg, double sy_arg, double2* __restrict__ Kp, double2* __restrict__ Wp, int p,
                   const Noise nz, double* nis_acc, double* nis_out, int nis_flags) {
    large_gain_p<NIS>(sig, ld, N, state_in, state_out, pose_src, cmd, lm_arg, sx_arg, sy_arg, Kp, Wp, p,
                      NOISE ? nz : ref_noise(), nis_acc, nis_out, nis_flags);
}

// prediction() with factors pending: Sigma' = A (Sigma_0 - sum_j K_j W_j) A^T + Q = [A Sigma_0 A^T + Q] - sum_j (A K_j)(W_j A^T)
// with A = I + a1 e1 e0^T + a2 e2 e0^T (ekf_slam.cpp:89-102).  The bracket is the usual strip update of the stored
// Sigma_0; the factors take K_j[1] += a1 K_j[0], K_j[2] += a2 K_j[0] and W_j[:,1] += a1 W_j[:,0], W_j[:,2] += a2 W_j[:,0]:
// O(1) per factor (lanes j < pending of k_large_motion), so the sweep does not have to run before every prediction and
// a group can span SLAM steps.

// Sigma[r][c] <- Sigma[r][c] - sum_{j<P} K_j[r] W_j[c], one pass over Sigma.  COLS columns per thread (4 -> 256-bit
// accesses, 2 -> 128-bit) so that the P x COLS W-pairs stay in registers for the whole tile.
template <int P, int COLS, int U, int ROWS, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
    k_large_sweep_p(double* __restrict__ sig, long long ld, int n_rows, const double2* __restrict__ Kp,
                    const double2* __restrict__ Wp, long long row0, unsigned long long* __restrict__ n_updates,
                    int n_counted, const UpdateCmd* __restrict__ cmd) {
    if (cmd && !cmd->do_update) return;  // association dropped the measurement: nothing to apply (P == 1 there)
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_updates) *n_updates += (unsigned long long)n_counted;
    constexpr int CHUNK = THREADS * COLS;
    const int chunks = (int)((ld + CHUNK - 1) / CHUNK);
    const int row_blocks = (n_rows + ROWS - 1) / ROWS;
    const long long tiles = (long long)chunks * row_blocks;
    for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int rb = (int)(t / chunks), cc = (int)(t - (long long)rb * chunks);
        const long long c = (long long)cc * CHUNK + threadIdx.x * COLS;
        if (c >= ld) continue;
        double2 w[P][COLS];
#pragma unroll
        for (int j = 0; j < P; ++j)
#pragma unroll
            for (int q = 0; q < COLS; ++q) w[j][q] = Wp[(long long)j * ld + c + q];
        const int r_begin = rb * ROWS;
        const int r_end = min(n_rows, r_begin + ROWS);
        double* ptr = sig + (long long)r_begin * ld + c;
        // U rows (U x 32 B of loads) in flight per thread
        int r = r_begin;
        for (; r + U <= r_end; r += U) {
            double v[U][COLS];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (COLS == 4) {
                    ld256(ptr + u * ld, v[u][0], v[u][1], v[u][2], v[u][3]);
                } else {
                    const double2 t2 = *reinterpret_cast<const double2*>(ptr + u * ld);
                    v[u][0] = t2.x;
                    v[u][1] = t2.y;
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
#pragma unroll
                for (int j = 0; j < P; ++j) {
                    const double2 k = Kp[(long long)j * ld + row0 + r + u];
#pragma unroll
                    for (int q = 0; q < COLS; ++q) v[u][q] = apply_factor(v[u][q], k, w[j][q]);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (COLS == 4) {
                    st256(ptr + u * ld, v[u][0], v[u][1], v[u][2], v[u][3]);
                } else {
                    *reinterpret_cast<double2*>(ptr + u * ld) = make_double2(v[u][0], v[u][1]);
                }
            }
            ptr += (long long)U * ld;
        }
        for (; r < r_end; ++r) {
            double v[COLS];
            if (COLS == 4) {
                ld256(ptr, v[0], v[1], v[2], v[3]);
            } else {
                const double2 t2 = *reinterpret_cast<const double2*>(ptr);
                v[0] = t2.x;
                v[1] = t2.y;
            }
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double2 k = Kp[(long long)j * ld + row0 + r];
#pragma unroll
                for (int q = 0; q < COLS; ++q) v[q] = apply_factor(v[q], k, w[j][q]);
            }
            if (COLS == 4) {
                st256(ptr, v[0], v[1], v[2], v[3]);
            } else {
                *reinterpret_cast<double2*>(ptr) = make_double2(v[0], v[1]);
            }
            ptr += ld;
        }
    }
}

// One CTA per tile (ROWS x THREADS*4 columns): on B200 the plain full grid beats a persistent grid-stride launch here
// (experiments/sweep_tune.cu: P=1 0.65 ms = 6.6 TB/s at N = 16,387; P=4..6 0.79-0.82 ms; P=8 0.98 ms — the FMAs of a
// tile do not overlap its own loads).  So the register path only serves 1-2 factors; deeper groups go to
// k_large_sweep_mma (ekf_large_mma.cuh).
template <int P, int U, int ROWS, int THREADS>
inline void launch_sweep_cfg(double* sig, long long ld, int n_rows, const double2* Kp, const double2* Wp, long long row0,
                             unsigned long long* n_updates, int n_counted, const UpdateCmd* cmd, cudaStream_t stream) {
    const long long chunk = (long long)THREADS * 4;
    const long long tiles = ((ld + chunk - 1) / chunk) * ((n_rows + ROWS - 1) / ROWS);
    k_large_sweep_p<P, 4, U, ROWS, THREADS><<<(unsigned)(tiles < 1 ? 1 : tiles), THREADS, 0, stream>>>(
        sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd);
}

inline cudaError_t launch_sweep_p(int pending, double* sig, long long ld, int n_rows, const double2* Kp, const double2* Wp,
                                  long long row0, unsigned long long* n_updates, int n_counted, const UpdateCmd* cmd,
                                  cudaStream_t stream) {
    switch (pending) {
        case 1: launch_sweep_cfg<1, 4, 32, 256>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, stream); break;
        case 2: launch_sweep_cfg<2, 4, 32, 256>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, stream); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace ekf
