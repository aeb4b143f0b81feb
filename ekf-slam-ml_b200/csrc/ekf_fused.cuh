// Engine 1: the whole EKF-SLAM step of one filter (prediction + measurement() or data_association())
// in ONE kernel, one warp per filter, with Sigma resident in shared memory for all of the step's
// sequential rank-2 updates.  Sigma and the state are staged HBM -> smem -> HBM with the bulk copy
// engine (TMA), so per filter and step HBM sees exactly one read and one write of Sigma, however many
// landmarks are corrected.  Used for the Monte-Carlo batch (B = 65,536 x n = 20) and, with B = 1, for a
// single reference-sized filter (one launch per API call instead of ~10 launches).
//
// Restates rigid2d/src/ekf_slam.cpp:55-106 (prediction), :108-197 (measurement), :200-214
// (initialize_landmark), :217-276 (calculate_maha_dis), :278-402 (data_association).
#pragma once
#include "bulk_copy.cuh"
#include "ekf_math.cuh"

namespace ekf {

enum FusedMode : int { kDoPredict = 1, kDoMeasurement = 2, kDoAssociation = 4, kSparseReadings = 8 };

struct FusedParams {
    double* sigma;         // [B][sig_stride]   row-major N x N per filter, stride padded to 16 doubles
    double* state;         // [B][st_stride]    theta, x, y, m1x, m1y, ...
    int32_t* init_flag;    // [B]               landmark_init_flag (ekf_slam.cpp:50)
    uint8_t* known;        // [B][n]            known_list (data_association only, in/out)
    const double* twists;  // [B][2]            {dtheta, dx}
    const double* xy;      // measurement: [B][2n] robot-frame readings; association: [B][m_max][2]
    const uint8_t* vis;    // [B][n]
    const int32_t* mcount; // [B]               number of valid measurements (association)
    int32_t* assoc_out;    // [B][m_max] or null
    double* dmin_out;      // [B][m_max] or null
    double* second_out;    // [B][m_max] or null
    uint8_t* created_out;  // [B][m_max] or null
    unsigned long long* n_updates;  // running count of landmark corrections, or null
    double* pose_out;      // [B][3] or null: theta, x, y after the step (single filter: mapped pinned host memory)
    long long B;
    int n;
    int m_max;
    int mode;
    int sig_stride;  // doubles
    int st_stride;   // doubles
    long long sparse_total;  // marker-list mode: number of listed markers (offsets are checked against it)
    double* nis;             // [B][4] NIS accumulators of the batch kernels' NIS variants (nis() / nis_add())
};

__host__ __device__ inline int fused_round16(int v) { return (v + 15) & ~15; }

// shared memory carve-up (bytes), identical on host and device
struct FusedSmem {
    int off_sig, off_st, off_k2, off_w2, off_k2b, off_w2b, off_z, off_bar, total;
    __host__ __device__ FusedSmem(int n, int m_max) {
        const int N = 3 + 2 * n;
        int o = 0;
        off_sig = o;
        o += fused_round16(N * N) * 8;
        off_st = o;
        o += fused_round16(N) * 8;
        off_k2 = o;  // factor A: K (N x 2) and W (2 x N) as double2 per row / column
        o += N * 16;
        off_w2 = o;
        o += N * 16;
        off_k2b = o;  // factor B (second correction of a pair)
        o += N * 16;
        off_w2b = o;
        o += N * 16;
        o = (o + 15) & ~15;
        off_z = o;
        const int zc = 2 * (n > m_max ? n : m_max);
        o += zc * 8;  // n = 20: 18,320 B per CTA in total, so that 12 CTAs (+1 KB reserve each) fit one SM's 227 KB
        off_bar = o;
        o += 16;
        total = o;
    }
};

__device__ __forceinline__ double apply_pair(double v, double2 k, double2 w) {
    return fma(-k.y, w.y, fma(-k.x, w.x, v));
}

// Gain part of one landmark correction on the smem-resident filter (ekf_slam.cpp:138-187 == :335-385):
// W = Hj Sigma (2 x N) -> Wout, K = Sigma Hj^T S^-1 (N x 2) -> Kout, state += K nu.  Sigma itself is NOT touched.
// If PEND, Sigma in shared memory is still missing the factor pair (Kpend, Wpend) of the previous correction; the
// five rows and five columns that this correction needs are rebuilt on the fly with exactly the FMAs the rank-2
// update would have applied (so the result is bit-identical to updating Sigma after every correction).
// All lanes enter with identical (i, h, zr, zphi); h = H_j / z_hat of landmark i from the current state.
template <bool PEND>
__device__ __forceinline__ void warp_gain(const double* __restrict__ sig, double* __restrict__ st,
                                          const double2* __restrict__ Kpend, const double2* __restrict__ Wpend,
                                          double2* __restrict__ Kout, double2* __restrict__ Wout, const int N,
                                          const int lane, const int i, const Hj h, const double zr, const double zphi) {
    const int i3 = 3 + 2 * i, i4 = i3 + 1;
    double2 ka[5], wa[5];
    if (PEND) {
        ka[0] = Kpend[0], ka[1] = Kpend[1], ka[2] = Kpend[2], ka[3] = Kpend[i3], ka[4] = Kpend[i4];
        wa[0] = Wpend[0], wa[1] = Wpend[1], wa[2] = Wpend[2], wa[3] = Wpend[i3], wa[4] = Wpend[i4];
    }
    // W = Hj * Sigma (from 5 rows) and P = Sigma * Hj^T (from 5 columns)
    for (int c = lane; c < N; c += 32) {
        double s0 = sig[c], s1 = sig[N + c], s2 = sig[2 * N + c];
        double s3 = sig[i3 * N + c], s4 = sig[i4 * N + c];
        const double* row = sig + c * N;
        double r0 = row[0], r1 = row[1], r2 = row[2], r3 = row[i3], r4 = row[i4];
        if (PEND) {
            const double2 wc = Wpend[c], kc = Kpend[c];
            s0 = apply_pair(s0, ka[0], wc);
            s1 = apply_pair(s1, ka[1], wc);
            s2 = apply_pair(s2, ka[2], wc);
            s3 = apply_pair(s3, ka[3], wc);
            s4 = apply_pair(s4, ka[4], wc);
            r0 = apply_pair(r0, kc, wa[0]);
            r1 = apply_pair(r1, kc, wa[1]);
            r2 = apply_pair(r2, kc, wa[2]);
            r3 = apply_pair(r3, kc, wa[3]);
            r4 = apply_pair(r4, kc, wa[4]);
        }
        Wout[c] = make_double2(h_row0(h, s1, s2, s3, s4), h_row1(h, s0, s1, s2, s3, s4));
        Kout[c] = make_double2(h_row0(h, r1, r2, r3, r4), h_row1(h, r0, r1, r2, r3, r4));
    }
    __syncwarp();
    // S = (Hj Sigma) Hj^T + R from W at the five columns; closed-form inverse
    const double2 w0 = Wout[0], w1 = Wout[1], w2 = Wout[2], w3 = Wout[i3], w4 = Wout[i4];
    const double s00 = h_row0(h, w1.x, w2.x, w3.x, w4.x) + kR;
    const double s01 = h_row1(h, w0.x, w1.x, w2.x, w3.x, w4.x);
    const double s10 = h_row0(h, w1.y, w2.y, w3.y, w4.y);
    const double s11 = h_row1(h, w0.y, w1.y, w2.y, w3.y, w4.y) + kR;
    const Sym2 si = inv2x2(s00, s01, s10, s11);
    const double nu0 = __dsub_rn(zr, h.zr);
    const double nu1 = normalize_angle(__dsub_rn(zphi, h.zphi));  // :182-183
    // K = P S^-1; state += K nu
    for (int r = lane; r < N; r += 32) {
        const double2 p = Kout[r];
        const double k0 = fma(p.y, si.i10, p.x * si.i00);
        const double k1 = fma(p.y, si.i11, p.x * si.i01);
        Kout[r] = make_double2(k0, k1);
        double ns = st[r] + fma(k1, nu1, k0 * nu0);
        if (r == 0) ns = normalize_angle(ns);  // theta is wrapped after every correction (:187)
        st[r] = ns;
    }
    __syncwarp();
}

// Sigma <- Sigma - Ka Wa [- Kb Wb]   ((I - K Hj) Sigma, ekf_slam.cpp:191-192, for one or two corrections in ONE pass
// over the shared-memory copy of Sigma; the factors are applied in order, two FMAs each, per element).
// Lane tiling 2 row groups x 16 column groups: lane (g, q) owns rows g, g+2, ... and columns q, q+16, q+32, ...
// Its W pairs stay in registers for the whole pass and each K pair is fetched once per row.  N is odd, so a
// half-warp (fixed g, q = 0..15) always hits 16 distinct 8-byte bank slots: conflict-free for every map size.
// Rows go through in batches of RB so that one shared-memory latency is paid per batch, not per row.
template <int NL, int NF>
__device__ __forceinline__ void warp_rank2(double* __restrict__ sig, const double2* __restrict__ Ka,
                                           const double2* __restrict__ Wa, const double2* __restrict__ Kb,
                                           const double2* __restrict__ Wb, const int N, const int lane) {
    constexpr int NC = NL ? 3 + 2 * NL : 0;
    const int g = lane >> 4, q = lane & 15;
    if (NC) {
        constexpr int CB = NC ? (NC + 15) / 16 : 1;  // column slots per lane
        constexpr int RA = NC ? (NC + 1) / 2 : 1;    // row slots per lane
        constexpr int RB = (NF == 1) ? 6 : 4;
        double2 wa[CB], wb[CB];
#pragma unroll
        for (int b = 0; b < CB; ++b) {
            wa[b] = (q + 16 * b < NC) ? Wa[q + 16 * b] : make_double2(0.0, 0.0);
            if (NF == 2) wb[b] = (q + 16 * b < NC) ? Wb[q + 16 * b] : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int a0 = 0; a0 < RA; a0 += RB) {
            double2 ka[RB], kb[RB];
            double v[RB][CB];
#pragma unroll
            for (int u = 0; u < RB; ++u) {
                const int r = g + 2 * (a0 + u);
                if (a0 + u < RA && r < NC) {
                    ka[u] = Ka[r];
                    if (NF == 2) kb[u] = Kb[r];
#pragma unroll
                    for (int b = 0; b < CB; ++b)
                        if (q + 16 * b < NC) v[u][b] = sig[r * NC + q + 16 * b];
                }
            }
#pragma unroll
            for (int u = 0; u < RB; ++u) {
                const int r = g + 2 * (a0 + u);
                if (a0 + u < RA && r < NC) {
#pragma unroll
                    for (int b = 0; b < CB; ++b)
                        if (q + 16 * b < NC) {
                            double t = apply_pair(v[u][b], ka[u], wa[b]);
                            if (NF == 2) t = apply_pair(t, kb[u], wb[b]);
                            sig[r * NC + q + 16 * b] = t;
                        }
                }
            }
        }
    } else {
        for (int c0 = 0; c0 < N; c0 += 64) {  // four column slots per pass keep the generic path in registers
            double2 wa[4], wb[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int c = c0 + q + 16 * b;
                wa[b] = c < N ? Wa[c] : make_double2(0.0, 0.0);
                if (NF == 2) wb[b] = c < N ? Wb[c] : make_double2(0.0, 0.0);
            }
            for (int r = g; r < N; r += 2) {
                const double2 ka = Ka[r];
                double2 kb = make_double2(0.0, 0.0);
                if (NF == 2) kb = Kb[r];
                double* row = sig + r * N + c0 + q;
#pragma unroll
                for (int b = 0; b < 4; ++b)
                    if (c0 + q + 16 * b < N) {
                        double t = apply_pair(row[16 * b], ka, wa[b]);
                        if (NF == 2) t = apply_pair(t, kb, wb[b]);
                        row[16 * b] = t;
                    }
            }
        }
    }
    __syncwarp();
}

// ---- shared by ekf_fused_kernel (dense Sigma) and ekf_fused_sym_kernel (staircase Sigma, ekf_fused_sym.cuh)

// Prediction (ekf_slam.cpp:55-106): Sigma <- A Sigma A^T + Q with A = I + a1 e1 e0^T + a2 e2 e0^T, and the state.
// Rows 1, 2 take a * row 0 over all N columns; columns 1, 2 take a * column 0 in the rows below col_rows: all N rows
// of a dense Sigma, the first diagonal block of the staircase (beyond it, columns 1, 2 ARE rows 1, 2).
__device__ __forceinline__ Motion fused_predict(double* sig, double* st, const int N, const int col_rows, const int lane,
                                                const double dtheta, const double dxv) {
    const Motion mo = motion_model(st[0], dtheta, dxv);
    __syncwarp();
    for (int c = lane; c < N; c += 32) {
        const double r0 = sig[c];
        sig[N + c] = fma(mo.a1, r0, sig[N + c]);
        sig[2 * N + c] = fma(mo.a2, r0, sig[2 * N + c]);
    }
    __syncwarp();
    for (int r = lane; r < col_rows; r += 32) {
        const double c0 = sig[r * N];
        sig[r * N + 1] = fma(c0, mo.a1, sig[r * N + 1]);
        sig[r * N + 2] = fma(c0, mo.a2, sig[r * N + 2]);
    }
    __syncwarp();
    if (lane == 0) {
        sig[0] += kQ;
        sig[N + 1] += kQ;
        sig[2 * N + 2] += kQ;
        st[0] = st[0] + mo.u0;  // theta is not wrapped here (:99)
        st[1] = st[1] + mo.u1;
        st[2] = st[2] + mo.u2;
    }
    __syncwarp();
    return mo;
}

// Inputs of data_association(), fetched while Sigma is still in flight: the number of readings, clamped to
// [0, m_max], and (range, bearing) of each reading in zbuf (ekf_slam.cpp:338-344).  Returns the count.
__device__ __forceinline__ int fused_assoc_inputs(const FusedParams& p, const long long b, const int lane, double* zbuf) {
    int m = p.mcount ? p.mcount[b] : p.m_max;
    m = m < 0 ? 0 : (m < p.m_max ? m : p.m_max);  // a negative count is an empty list
    for (int j = lane; j < m; j += 32) {
        const double sx = p.xy[(b * p.m_max + j) * 2], sy = p.xy[(b * p.m_max + j) * 2 + 1];
        double r, phi;
        range_bearing(sx, sy, r, phi);
        zbuf[2 * j] = r;
        zbuf[2 * j + 1] = phi;
    }
    return m;
}

// data_association(): Mahalanobis nearest neighbour + landmark initialisation (ekf_slam.cpp:278-402) for the m
// readings in zbuf.  The Sigma layout enters through two calls only:
//   dist(i, zr, zphi, theta, x, y)  distance of known landmark i (each lane scans its own landmarks);
//   correct(i, h, zr, zphi, created) gain, state update and rank-2 update of landmark i (whole warp; h from the live
//                                    pose); `created` is set when this very reading initialised the landmark.
template <class Dist, class Correct>
__device__ __forceinline__ void fused_association(const FusedParams& p, const long long b, const int n, const int m,
                                                  const int lane, double* st, const double* zbuf,
                                                  unsigned long long& n_corr, Dist dist, Correct correct) {
    uint8_t* known = p.known + b * n;
    int known_count = 0;  // leading-true prefix (:281-288)
    for (int base = 0; base < n; base += 32) {
        const int i_l = base + lane;
        const unsigned ones = __ballot_sync(0xffffffffu, i_l < n && known[i_l] != 0);
        const int lead = __ffs(~ones) - 1;  // number of leading ones in this group of 32 (32 -> -1)
        if (ones == 0xffffffffu) {
            known_count += 32;
            continue;
        }
        known_count += lead;
        break;
    }
    if (known_count > n) known_count = n;
    const int known_count0 = known_count;
    for (int j = 0; j < m; ++j) {
        const double zr = zbuf[2 * j], zphi = zbuf[2 * j + 1];
        const double theta = st[0], x = st[1], y = st[2];  // live pose (:219-221)
        double best = INFINITY, second = INFINITY;
        int best_i = 0x7fffffff;
        for (int i = lane; i < known_count; i += 32) {
            double d = dist(i, zr, zphi, theta, x, y);
            if (!(d == d)) d = INFINITY;  // NaN never wins
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
            if (better(ob, oi, best, best_i)) {
                second = fmin(best, os);
                best = ob;
                best_i = oi;
            } else {
                second = fmin(second, ob);
            }
        }
        double min_d = kGateNew;
        int min_idx = known_count;
        if (best < kGateNew) {  // d < min_maha_dis, :305
            min_d = best;
            min_idx = best_i;
            second = fmin(second, kGateNew);
        } else {
            second = best;
        }
        const long long o = b * p.m_max + j;
        if (lane == 0) {
            if (p.dmin_out) p.dmin_out[o] = min_d;
            if (p.second_out) p.second_out[o] = second;
        }
        int created = 0;
        if (min_idx == known_count && min_idx < n) {  // :318-327
            if (lane == 0) {  // inline: an out-of-line call here would cost ekf_fused_kernel stack for its registers
                double mx, my;
                landmark_from_reading(p.xy[o * 2], p.xy[o * 2 + 1], theta, x, y, mx, my);
                st[3 + 2 * min_idx] = mx;
                st[4 + 2 * min_idx] = my;
            }
            __syncwarp();
            known_count++;
            min_d = 0.0;
            created = 1;
        }
        int assoc = -1;
        if (min_d < kGateUpdate) {  // :330
            const double th_l = st[0], x_l = st[1], y_l = st[2];  // live pose (:331-333)
            const Hj h = make_hj(st[3 + 2 * min_idx], st[4 + 2 * min_idx], th_l, x_l, y_l);
            correct(min_idx, h, zr, zphi, created);  // the next distances need the new Sigma
            ++n_corr;
            assoc = min_idx;
        }
        if (lane == 0) {
            if (p.assoc_out) p.assoc_out[o] = assoc;
            if (p.created_out) p.created_out[o] = (uint8_t)created;
        }
    }
    for (int i = known_count0 + lane; i < known_count; i += 32) known[i] = 1;
    if (lane == 0) {  // outputs beyond the valid count are defined too
        for (int j = m; j < p.m_max; ++j) {
            const long long o = b * p.m_max + j;
            if (p.assoc_out) p.assoc_out[o] = -1;
            if (p.created_out) p.created_out[o] = 0;
            if (p.dmin_out) p.dmin_out[o] = kGateNew;
            if (p.second_out) p.second_out[o] = INFINITY;
        }
    }
}

template <int NL>
__global__ void __launch_bounds__(32) ekf_fused_kernel(const FusedParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int n = NL ? NL : p.n;
    const int N = 3 + 2 * n;
    const FusedSmem L(n, p.m_max);
    double* sig = reinterpret_cast<double*>(smem_raw + L.off_sig);
    double* st = reinterpret_cast<double*>(smem_raw + L.off_st);
    double2* K2 = reinterpret_cast<double2*>(smem_raw + L.off_k2);
    double2* W2 = reinterpret_cast<double2*>(smem_raw + L.off_w2);
    double2* K2b = reinterpret_cast<double2*>(smem_raw + L.off_k2b);
    double2* W2b = reinterpret_cast<double2*>(smem_raw + L.off_w2b);
    double* zbuf = reinterpret_cast<double*>(smem_raw + L.off_z);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);

    const int lane = threadIdx.x;
    const long long b = blockIdx.x;
    if (b >= p.B) return;
    double* g_sig = p.sigma + b * (long long)p.sig_stride;
    double* g_st = p.state + b * (long long)p.st_stride;
    const uint32_t sig_bytes = (uint32_t)p.sig_stride * 8u, st_bytes = (uint32_t)p.st_stride * 8u;

    // ---- stage Sigma and the state into shared memory with the bulk copy engine
    if (lane == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
        mbar_arrive_expect_tx(bar, sig_bytes + st_bytes);
        bulk_g2s(sig, g_sig, sig_bytes, bar);
        bulk_g2s(st, g_st, st_bytes, bar);
    }
    // inputs that do not depend on the filter state are fetched while the copy is in flight
    double dtheta = 0.0, dxv = 0.0;
    if (p.mode & kDoPredict) {
        dtheta = p.twists[2 * b];
        dxv = p.twists[2 * b + 1];
    }
    int init_flag = p.init_flag[b];
    int m = 0;
    if (p.mode & kDoMeasurement) {
        // z = (range, bearing) of every slot's reading, lane-parallel (ekf_slam.cpp:140-146)
        for (int i = lane; i < n; i += 32) {
            const double sx = p.xy[b * 2 * n + 2 * i], sy = p.xy[b * 2 * n + 2 * i + 1];
            double r, phi;
            range_bearing(sx, sy, r, phi);
            zbuf[2 * i] = r;
            zbuf[2 * i + 1] = phi;
        }
    } else if (p.mode & kDoAssociation) {
        m = fused_assoc_inputs(p, b, lane, zbuf);
    }
    __syncwarp();
    mbar_wait(bar, 0);

    // ---- prediction (ekf_slam.cpp:55-106)
    if (p.mode & kDoPredict) fused_predict(sig, st, N, N, lane, dtheta, dxv);

    unsigned long long n_corr = 0;

    // ---- measurement(): known association (ekf_slam.cpp:108-197)
    if (p.mode & kDoMeasurement) {
        const double theta = st[0], x = st[1], y = st[2];  // read once; stale for later i (:109-111)
        if (!init_flag) {
            for (int i = lane; i < n; i += 32) {
                double mx, my;
                landmark_from_reading(p.xy[b * 2 * n + 2 * i], p.xy[b * 2 * n + 2 * i + 1], theta, x, y, mx, my);
                st[3 + 2 * i] = mx;
                st[4 + 2 * i] = my;
            }
            init_flag = 1;
            __syncwarp();
        }
        const uint8_t* vis = p.vis + b * n;
        for (int base = 0; base < n; base += 32) {
            const int i_l = base + lane;
            const unsigned mask = __ballot_sync(0xffffffffu, i_l < n && vis[i_l] != 0);
            // Visible landmarks go through in PAIRS: both gains are computed first (the second one sees the first
            // one's factor as "pending"), then ONE pass over Sigma applies both rank-2 updates.  That halves the
            // shared-memory traffic of the covariance update, which is what bounds this kernel.  H_j of the next
            // landmark is always evaluated right after the state update it depends on and before the covariance pass,
            // so the long scalar chain overlaps the pass's shared-memory latency.
            unsigned rem = mask;
            Hj h;
            if (rem) {
                const int i0 = base + __ffs(rem) - 1;
                h = make_hj(st[3 + 2 * i0], st[4 + 2 * i0], theta, x, y);
            }
            while (rem) {
                const int ia = base + __ffs(rem) - 1;
                rem &= rem - 1;
                warp_gain<false>(sig, st, nullptr, nullptr, K2, W2, N, lane, ia, h, zbuf[2 * ia], zbuf[2 * ia + 1]);
                ++n_corr;
                if (rem) {
                    const int ib = base + __ffs(rem) - 1;
                    rem &= rem - 1;
                    h = make_hj(st[3 + 2 * ib], st[4 + 2 * ib], theta, x, y);
                    warp_gain<true>(sig, st, K2, W2, K2b, W2b, N, lane, ib, h, zbuf[2 * ib], zbuf[2 * ib + 1]);
                    ++n_corr;
                    if (rem) {
                        const int in = base + __ffs(rem) - 1;
                        h = make_hj(st[3 + 2 * in], st[4 + 2 * in], theta, x, y);
                    }
                    warp_rank2<NL, 2>(sig, K2, W2, K2b, W2b, N, lane);
                } else {
                    warp_rank2<NL, 1>(sig, K2, W2, nullptr, nullptr, N, lane);
                }
            }
        }
    }

    // ---- data_association(): Mahalanobis nearest neighbour + landmark initialisation (ekf_slam.cpp:278-402)
    if (p.mode & kDoAssociation) {
        fused_association(
            p, b, n, m, lane, st, zbuf, n_corr,
            [&](int i, double zr, double zphi, double theta, double x, double y) {
                return maha_distance(sig, N, i, st[3 + 2 * i], st[4 + 2 * i], zr, zphi, theta, x, y);
            },
            [&](int i, const Hj& h, double zr, double zphi, int) {
                warp_gain<false>(sig, st, nullptr, nullptr, K2, W2, N, lane, i, h, zr, zphi);
                warp_rank2<NL, 1>(sig, K2, W2, nullptr, nullptr, N, lane);
            });
    }

    // ---- write back: smem -> HBM with the bulk copy engine
    __syncwarp();
    fence_proxy_async_smem();
    __syncwarp();
    if (p.pose_out && lane < 3) p.pose_out[3 * b + lane] = st[lane];
    if (lane == 0) {
        bulk_s2g(g_sig, sig, sig_bytes);
        bulk_s2g(g_st, st, st_bytes);
        bulk_commit();
        p.init_flag[b] = init_flag;
        if (p.n_updates && n_corr) atomicAdd(p.n_updates, n_corr);
        bulk_wait_all();
    }
}

}  // namespace ekf
