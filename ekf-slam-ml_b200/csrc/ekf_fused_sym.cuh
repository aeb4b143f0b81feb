// Engine 1b: the batched fused step with Sigma kept SYMMETRIC in a block-staircase layout.
//
// Same step as ekf_fused.cuh (prediction + measurement() or data_association() of one filter per warp, Sigma
// resident in shared memory, staged by the bulk copy engine), but only the block-upper part of Sigma exists, in HBM
// and on chip: row r keeps the columns [16*floor(r/16), N).  For N = 43 that is 1,241 of 1,849 entries, which
//   * cuts the shared memory per filter from 18.3 KB to 13.5 KB -> 16 resident filters per SM instead of 12,
//   * cuts the rank-2 pass (the (I - K H) Sigma of ekf_slam.cpp:191-192) to the stored entries (46 instead of 66
//     half-warp tiles per factor) and the gain to five row reads (K = (H Sigma)^T S^-1, no column reads),
//   * cuts the HBM traffic per filter-step by the same third.
// Every row stride (N - 16 rb) is odd, so row reads, transposed reads and the 2 x 16 tiles are bank-conflict free.
// Mathematically Sigma stays symmetric under both the prediction and the correction; the reference's dense
// products leave rounding-level asymmetry (1e-16 relative) that this layout does not carry, far inside the 1e-9
// parity tolerance.  Entries below the diagonal inside a diagonal block are stored and updated like any other.
//
// Restates rigid2d/src/ekf_slam.cpp:55-106, :108-197, :200-214, :217-276, :278-402 (as ekf_fused.cuh).
#pragma once
#include "ekf_fused.cuh"

namespace ekf {

// ---- staircase layout -------------------------------------------------------------------------------------------
// offset of element (r, 16*floor(r/16)) = start of the stored part of row r
__host__ __device__ constexpr int stair_row_base(int r, int N) {
    const int rb = r >> 4;
    return 16 * rb * N - 128 * rb * (rb - 1) + (r - 16 * rb) * (N - 16 * rb);
}
__host__ __device__ constexpr int stair_size(int N) { return stair_row_base(N, N); }
// offset of element (r, c) for any r, c (the mirror entry is used below the stored part)
__host__ __device__ __forceinline__ int stair_at(int r, int c, int N) {
    const bool t = c < (r & ~15);
    const int rr = t ? c : r, cc = t ? r : c;
    return stair_row_base(rr, N) + cc - (rr & ~15);
}

// per-filter strides (doubles) of the batch's Sigma and state arrays: multiples of 16 B for the bulk copies
__host__ __device__ constexpr int sym_sig_stride(int N) { return (stair_size(N) + 1) & ~1; }
__host__ __device__ constexpr int sym_st_stride(int N) { return (N + 1) & ~1; }

struct SymSmem {
    int off_sig, off_st, off_k2, off_w2, off_k2b, off_w2b, off_z, off_bar, off_nis, total;
    __host__ __device__ SymSmem(int n, int m_max, bool nis = false) {
        const int N = 3 + 2 * n;
        int o = 0;
        off_sig = o;
        o += sym_sig_stride(N) * 8;
        off_st = o;
        o += sym_st_stride(N) * 8;
        off_k2 = o;
        o += N * 16;
        off_w2 = o;
        o += N * 16;
        off_k2b = o;
        o += N * 16;
        off_w2b = o;
        o += N * 16;
        o = (o + 15) & ~15;
        off_z = o;
        const int zc = 3 * (n > m_max ? n : m_max);  // Reading {zr, ux, uy} per slot
        o += zc * 8;  // n = 20: 13,536 B per CTA: 16 CTAs of 13,568 B (+1 KB reserve each) fit one SM's 228 KB
        off_bar = o;
        o += 16;
        off_nis = o;  // NIS only: the step's sums {sum, sum^2, #scored, #non-finite}, kept by lane 0
        o += nis ? 4 * 8 : 0;
        total = o;
    }
};

constexpr int kSymSlots = 5;  // column slots per lane (n <= 64 -> N <= 131)

// Gain of one correction from five ROWS of the symmetric Sigma: W = Hj Sigma -> Wout, K = W^T S^-1 -> Kout,
// state += K nu.  With PEND the stored Sigma still misses the previous correction's factor (Kpend, Wpend); the
// entries read here are rebuilt with the FMAs the rank-2 pass will apply to them (in their stored orientation).
// cmv[s] = offset of the mirror row of the lane's column slot s (loop invariant, computed once per launch).  Returns
// S^-1 (warp-uniform) for the NIS of the correction.
template <bool PEND, class H>
__device__ __forceinline__ Sym2 sym_warp_gain(const double* __restrict__ sig, double* __restrict__ st,
                                              const double2* __restrict__ Kpend, const double2* __restrict__ Wpend,
                                              double2* __restrict__ Kout, double2* __restrict__ Wout, const int N,
                                              const int lane, const int* __restrict__ cmv, const int i, const H h,
                                              const double nu0, const double nu1) {
    const int i3 = 3 + 2 * i, i4 = i3 + 1;
    const int b3 = i3 & ~15, b4 = i4 & ~15;
    // row offsets of the landmark's two rows: lane r % 32 already holds stair_row_base(r) - (r & ~15) in cmv[r / 32]
    int row3 = __shfl_sync(0xffffffffu, cmv[0], i3 & 31), row4 = __shfl_sync(0xffffffffu, cmv[0], i4 & 31);
#pragma unroll
    for (int sl = 1; sl < kSymSlots; ++sl) {
        const int r3 = __shfl_sync(0xffffffffu, cmv[sl], i3 & 31), r4 = __shfl_sync(0xffffffffu, cmv[sl], i4 & 31);
        if ((i3 >> 5) == sl) row3 = r3;
        if ((i4 >> 5) == sl) row4 = r4;
    }
    double2 ka[5], wa3, wa4;
    if (PEND) {
        ka[0] = Kpend[0], ka[1] = Kpend[1], ka[2] = Kpend[2], ka[3] = Kpend[i3], ka[4] = Kpend[i4];
        wa3 = Wpend[i3], wa4 = Wpend[i4];
    }
    double2 wreg[kSymSlots];  // this lane's W columns stay in registers for the K loop
#pragma unroll
    for (int sl = 0; sl < kSymSlots; ++sl) {
        const int c = lane + 32 * sl;
        if (c < N) {
            const int cm = cmv[sl];
            const bool t3 = c < b3, t4 = c < b4;
            double s0 = sig[c], s1 = sig[N + c], s2 = sig[2 * N + c];
            double s3 = sig[t3 ? cm + i3 : row3 + c];
            double s4 = sig[t4 ? cm + i4 : row4 + c];
            if (PEND) {
                const double2 wc = Wpend[c], kc = Kpend[c];
                s0 = apply_pair(s0, ka[0], wc);
                s1 = apply_pair(s1, ka[1], wc);
                s2 = apply_pair(s2, ka[2], wc);
                s3 = apply_pair(s3, t3 ? kc : ka[3], t3 ? wa3 : wc);
                s4 = apply_pair(s4, t4 ? kc : ka[4], t4 ? wa4 : wc);
            }
            h_rows(h, s0, s1, s2, s3, s4, wreg[sl].x, wreg[sl].y);
            Wout[c] = wreg[sl];
        }
    }
    __syncwarp();
    // S = (Hj Sigma) Hj^T + R from W at the five columns; closed-form inverse
    const double2 w0 = Wout[0], w1 = Wout[1], w2 = Wout[2], w3 = Wout[i3], w4 = Wout[i4];
    double s00, s01, s10, s11;
    h_rows(h, w0.x, w1.x, w2.x, w3.x, w4.x, s00, s01);
    h_rows(h, w0.y, w1.y, w2.y, w3.y, w4.y, s10, s11);
    const Sym2 si = inv2x2(s00 + kR, s01, s10, s11 + kR);
    // K = W^T S^-1 folded with nu: state += K nu
#pragma unroll
    for (int sl = 0; sl < kSymSlots; ++sl) {
        const int r = lane + 32 * sl;
        if (r < N) {
            const double2 p = wreg[sl];
            const double k0 = fma(p.y, si.i10, p.x * si.i00);
            const double k1 = fma(p.y, si.i11, p.x * si.i01);
            double ns = st[r] + fma(k1, nu1, k0 * nu0);
            if (r == 0) ns = normalize_angle(ns);  // theta is wrapped after every correction (:187)
            Kout[r] = make_double2(k0, k1);
            st[r] = ns;
        }
    }
    __syncwarp();
    return si;
}

// Sigma <- Sigma - Ka Wa [- Kb Wb] over the stored entries, block row by block row (rows 16 rb .. 16 rb + 15,
// columns from 16 rb on).  Lane (g, q) = (lane / 16, lane % 16) owns rows of parity g and the columns q + 16 b.
template <int NF>
__device__ __forceinline__ void sym_warp_rank2(double* __restrict__ sig, const double2* __restrict__ Ka,
                                               const double2* __restrict__ Wa, const double2* __restrict__ Kb,
                                               const double2* __restrict__ Wb, const int N, const int lane) {
    const int g = lane >> 4, q = lane & 15;
    const int nbk = (N + 15) >> 4;
    for (int rb = 0; rb < nbk; ++rb) {
        const int L = N - 16 * rb, rows = L < 16 ? L : 16, base = stair_row_base(16 * rb, N);
        for (int c0 = 0; c0 < L; c0 += 64) {  // four column slots per pass keep the W pairs in registers
            double2 wa[4], wb[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int c = 16 * rb + c0 + q + 16 * b;
                wa[b] = c < N ? Wa[c] : make_double2(0.0, 0.0);
                wb[b] = (NF == 2 && c < N) ? Wb[c] : make_double2(0.0, 0.0);
            }
            for (int lr = g; lr < rows; lr += 2) {
                const double2 ka = Ka[16 * rb + lr];
                double2 kb = make_double2(0.0, 0.0);
                if (NF == 2) kb = Kb[16 * rb + lr];
                double* row = sig + base + lr * L + c0 + q;
#pragma unroll
                for (int b = 0; b < 4; ++b)
                    if (c0 + q + 16 * b < L) {
                        double t = apply_pair(row[16 * b], ka, wa[b]);
                        if (NF == 2) t = apply_pair(t, kb, wb[b]);
                        row[16 * b] = t;
                    }
            }
        }
    }
    __syncwarp();
}

// Mahalanobis distance from the 5 x 5 block Sigma[idx, idx], idx = {0, 1, 2, 3+2i, 4+2i} (ekf_slam.cpp:217-276; see
// maha_distance_rows).  The block is symmetric: 15 distinct entries, of which the robot's 3 x 3 corner `rob`
// (00 01 02 11 12 22) is the same for every landmark and is fetched once per measurement by the caller.
__device__ __forceinline__ double sym_maha_distance(const double* __restrict__ sig, int N, int i, const double* rob,
                                                    double mx, double my, double zr, double zphi, double theta,
                                                    double x, double y) {
    const Hj h = make_hj(mx, my, theta, x, y);
    const int i3 = 3 + 2 * i, i4 = i3 + 1;
    const int rb3 = stair_row_base(i3, N) - (i3 & ~15), rb4 = stair_row_base(i4, N) - (i4 & ~15);
    const double c03 = sig[i3], c04 = sig[i4], c13 = sig[N + i3], c14 = sig[N + i4], c23 = sig[2 * N + i3],
                 c24 = sig[2 * N + i4];
    const double l33 = sig[rb3 + i3], l34 = sig[rb3 + i4], l44 = sig[rb4 + i4];
    const double blk[5][5] = {{rob[0], rob[1], rob[2], c03, c04},
                              {rob[1], rob[3], rob[4], c13, c14},
                              {rob[2], rob[4], rob[5], c23, c24},
                              {c03, c13, c23, l33, l34},
                              {c04, c14, c24, l34, l44}};
    double wl0[5], wl1[5];
#pragma unroll
    for (int l = 0; l < 5; ++l) h_rows(h, blk[0][l], blk[1][l], blk[2][l], blk[3][l], blk[4][l], wl0[l], wl1[l]);
    double p00, p01, p10, p11;
    h_rows(h, wl0[0], wl0[1], wl0[2], wl0[3], wl0[4], p00, p01);
    h_rows(h, wl1[0], wl1[1], wl1[2], wl1[3], wl1[4], p10, p11);
    const Sym2 pi = inv2x2(p00 + kR, p01, p10, p11 + kR);
    const double v0 = __dsub_rn(zr, h.zr), v1 = __dsub_rn(zphi, h.zphi);
    const double t0 = __dadd_rn(__dmul_rn(v0, pi.i00), __dmul_rn(v1, pi.i10));
    const double t1 = __dadd_rn(__dmul_rn(v0, pi.i01), __dmul_rn(v1, pi.i11));
    return __dadd_rn(__dmul_rn(t0, v0), __dmul_rn(t1, v1));
}

// first-call / new-landmark initialisation happens once per landmark: keep its atan2 + sincos out of the hot code
static __device__ __noinline__ void landmark_from_reading_cold(double sx, double sy, double theta, double x, double y,
                                                               double& mx, double& my) {
    landmark_from_reading(sx, sy, theta, x, y, mx, my);
}

// NIS: also accumulate the NIS of the step's scored corrections into p.nis[b]; lane 0 keeps the running sums in shared
// memory, not in registers.
template <bool NIS>
__global__ void __launch_bounds__(32) ekf_fused_sym_kernel(const FusedParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int n = p.n;
    const int N = 3 + 2 * n;
    const SymSmem L(n, p.m_max, NIS);
    double* sig = reinterpret_cast<double*>(smem_raw + L.off_sig);
    double* st = reinterpret_cast<double*>(smem_raw + L.off_st);
    double2* K2 = reinterpret_cast<double2*>(smem_raw + L.off_k2);
    double2* W2 = reinterpret_cast<double2*>(smem_raw + L.off_w2);
    double2* K2b = reinterpret_cast<double2*>(smem_raw + L.off_k2b);
    double2* W2b = reinterpret_cast<double2*>(smem_raw + L.off_w2b);
    double* zbuf = reinterpret_cast<double*>(smem_raw + L.off_z);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);
    double* nacc = reinterpret_cast<double*>(smem_raw + L.off_nis);

    const int lane = threadIdx.x;
    const long long b = blockIdx.x;
    if (b >= p.B) return;
    double* g_sig = p.sigma + b * (long long)p.sig_stride;
    double* g_st = p.state + b * (long long)p.st_stride;
    const uint32_t sig_bytes = (uint32_t)p.sig_stride * 8u, st_bytes = (uint32_t)p.st_stride * 8u;
    if (NIS && lane == 0) nacc[0] = nacc[1] = nacc[2] = nacc[3] = 0.0;

    int cmv[kSymSlots];  // mirror-row offsets of this lane's column slots (see sym_warp_gain)
#pragma unroll
    for (int sl = 0; sl < kSymSlots; ++sl) {
        const int c = lane + 32 * sl;
        cmv[sl] = stair_row_base(c, N) - (c & ~15);
    }

    // ---- stage Sigma (staircase) and the state into shared memory with the bulk copy engine
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
    // visible landmarks as warp-uniform bit masks (slots 0..31 and 32..63), readings as {zr, ux, uy} per slot
    unsigned vismask[2] = {0u, 0u};
    int sp_begin = 0, sp_count = 0;
    if ((p.mode & kDoMeasurement) && (p.mode & kSparseReadings)) {
        // marker list: p.mcount = CSR offsets [B + 1], p.vis = landmark ids, p.xy = (x, y) per listed marker
        sp_begin = p.mcount[b];
        sp_count = p.mcount[b + 1] - sp_begin;
        // malformed offsets must not turn into out-of-bounds reads: such a filter gets an empty list
        if (sp_begin < 0 || sp_count < 0 || (long long)sp_begin + sp_count > p.sparse_total) sp_count = 0;
        for (int k0 = 0; k0 < sp_count; k0 += 32) {
            const int k = k0 + lane;
            const bool on = k < sp_count;
            int id = 0;
            if (on) {
                id = p.vis[sp_begin + k];
                const Reading z = make_reading(p.xy[2 * (long long)(sp_begin + k)], p.xy[2 * (long long)(sp_begin + k) + 1]);
                if (id < n) {
                    zbuf[3 * id] = z.zr;
                    zbuf[3 * id + 1] = z.ux;
                    zbuf[3 * id + 2] = z.uy;
                }
            }
            vismask[0] |= __reduce_or_sync(0xffffffffu, (on && id < 32 && id < n) ? 1u << id : 0u);
            vismask[1] |= __reduce_or_sync(0xffffffffu, (on && id >= 32 && id < n) ? 1u << (id - 32) : 0u);
        }
    } else if (p.mode & kDoMeasurement) {
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            vismask[base >> 5] = __ballot_sync(0xffffffffu, i < n && p.vis[b * n + i] != 0);
        }
        // range and unit direction of every slot's reading, lane-parallel (ekf_slam.cpp:140-146)
        for (int i = lane; i < n; i += 32) {
            const Reading z = make_reading(p.xy[b * 2 * n + 2 * i], p.xy[b * 2 * n + 2 * i + 1]);
            zbuf[3 * i] = z.zr;
            zbuf[3 * i + 1] = z.ux;
            zbuf[3 * i + 2] = z.uy;
        }
    } else if (p.mode & kDoAssociation) {
        m = fused_assoc_inputs(p, b, lane, zbuf);
    }
    __syncwarp();
    mbar_wait(bar, 0);

    // ---- prediction (ekf_slam.cpp:55-106): rows 1, 2 are stored in full (block row 0); columns 1, 2 exist as such
    // only inside the first diagonal block
    double sth = 0.0, cth = 1.0;
    bool have_sincos = false;
    if (p.mode & kDoPredict) {
        const Motion mo = fused_predict(sig, st, N, N < 16 ? N : 16, lane, dtheta, dxv);
        sth = mo.s_new, cth = mo.c_new, have_sincos = true;
    }

    unsigned long long n_corr = 0;

    // ---- measurement(): known association (ekf_slam.cpp:108-197)
    if (p.mode & kDoMeasurement) {
        const double theta = st[0], x = st[1], y = st[2];  // read once; stale for later i (:109-111)
        const bool score = init_flag != 0;  // the first call's readings initialised every landmark: nu ~ 0
        if (!init_flag) {
            if (p.mode & kSparseReadings) {
                // unlisted slots read (0, 0): the landmark starts at the robot's position, as with dense zeros
                for (int i = lane; i < n; i += 32) {
                    st[3 + 2 * i] = x;
                    st[4 + 2 * i] = y;
                }
                __syncwarp();
                for (int k = lane; k < sp_count; k += 32) {
                    const int id = p.vis[sp_begin + k];
                    if (id < n) {
                        double mx, my;
                        landmark_from_reading_cold(p.xy[2 * (long long)(sp_begin + k)], p.xy[2 * (long long)(sp_begin + k) + 1],
                                              theta, x, y, mx, my);
                        st[3 + 2 * id] = mx;
                        st[4 + 2 * id] = my;
                    }
                }
            } else {
                for (int i = lane; i < n; i += 32) {
                    double mx, my;
                    landmark_from_reading_cold(p.xy[b * 2 * n + 2 * i], p.xy[b * 2 * n + 2 * i + 1], theta, x, y, mx, my);
                    st[3 + 2 * i] = mx;
                    st[4 + 2 * i] = my;
                }
            }
            init_flag = 1;
            __syncwarp();
        }
        if (!have_sincos) sincos(theta, &sth, &cth);
        for (int base = 0; base < n; base += 32) {
            unsigned rem = vismask[base >> 5];
            // Visible landmarks go through in PAIRS: both gains first (the second sees the first one's factor as
            // pending), then ONE pass over Sigma applies both rank-2 updates.  H_j / nu of the next landmark are
            // evaluated right after the state update they depend on and before the pass, so the scalar chain
            // overlaps the pass's shared-memory latency.
            Innov h;
            if (rem) {
                const int i0 = base + __ffs(rem) - 1;
                h = make_innov(st[3 + 2 * i0], st[4 + 2 * i0], theta, sth, cth, x, y,
                               Reading{zbuf[3 * i0], zbuf[3 * i0 + 1], zbuf[3 * i0 + 2]});
            }
            bool second = false;
            while (rem) {
                const int ic = base + __ffs(rem) - 1;
                rem &= rem - 1;
                Sym2 si;
                if (!second)
                    si = sym_warp_gain<false>(sig, st, nullptr, nullptr, K2, W2, N, lane, cmv, ic, h, h.nu0, h.nu1);
                else
                    si = sym_warp_gain<true>(sig, st, K2, W2, K2b, W2b, N, lane, cmv, ic, h, h.nu0, h.nu1);
                if (NIS && score && lane == 0) nis_add(nacc, nis(si, h.nu0, h.nu1));
                ++n_corr;
                if (rem) {
                    const int in = base + __ffs(rem) - 1;
                    h = make_innov(st[3 + 2 * in], st[4 + 2 * in], theta, sth, cth, x, y,
                                   Reading{zbuf[3 * in], zbuf[3 * in + 1], zbuf[3 * in + 2]});
                }
                if (second)
                    sym_warp_rank2<2>(sig, K2, W2, K2b, W2b, N, lane);
                else if (!rem)
                    sym_warp_rank2<1>(sig, K2, W2, nullptr, nullptr, N, lane);
                second = !second;
            }
        }
    }

    // ---- data_association(): Mahalanobis nearest neighbour + landmark initialisation (ekf_slam.cpp:278-402)
    if (p.mode & kDoAssociation) {
        fused_association(
            p, b, n, m, lane, st, zbuf, n_corr,
            [&](int i, double zr, double zphi, double theta, double x, double y) {
                const double rob[6] = {sig[0], sig[1], sig[2], sig[N + 1], sig[N + 2], sig[2 * N + 2]};
                return sym_maha_distance(sig, N, i, rob, st[3 + 2 * i], st[4 + 2 * i], zr, zphi, theta, x, y);
            },
            [&](int i, const Hj& h, double zr, double zphi, int created) {
                const double nu0 = __dsub_rn(zr, h.zr), nu1 = normalize_angle(__dsub_rn(zphi, h.zphi));  // :182-183
                const Sym2 si = sym_warp_gain<false>(sig, st, nullptr, nullptr, K2, W2, N, lane, cmv, i, h, nu0, nu1);
                if (NIS && !created && lane == 0) nis_add(nacc, nis(si, nu0, nu1));  // a new landmark starts at its reading
                sym_warp_rank2<1>(sig, K2, W2, nullptr, nullptr, N, lane);
            });
    }

    // ---- write back: smem -> HBM with the bulk copy engine
    __syncwarp();
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
        bulk_s2g(g_sig, sig, sig_bytes);
        bulk_s2g(g_st, st, st_bytes);
        bulk_commit();
        p.init_flag[b] = init_flag;
        if (p.n_updates && n_corr) atomicAdd(p.n_updates, n_corr);
        if (NIS) {
#pragma unroll
            for (int k = 0; k < 4; ++k) p.nis[4 * b + k] += nacc[k];
        }
        bulk_wait_read();  // shared memory must outlive the copy engine's reads; the writes drain with the grid
    }
}

// Sigma_0 = blockdiag(0_3, 100 I) in the staircase layout (ekf_slam.cpp:36-47), zero state, init flag cleared.
__global__ void k_fused_sym_init(double* sigma, double* state, int32_t* init_flag, long long B, int N, int sig_stride,
                                 int st_stride) {
    const long long b = blockIdx.x;
    if (b >= B) return;
    double* s = sigma + b * (long long)sig_stride;
    for (int e = threadIdx.x; e < sig_stride; e += blockDim.x) s[e] = 0.0;
    __syncthreads();
    for (int r = 3 + threadIdx.x; r < N; r += blockDim.x) s[stair_at(r, r, N)] = kSigma0;
    for (int e = threadIdx.x; e < st_stride; e += blockDim.x) state[b * (long long)st_stride + e] = 0.0;
    if (threadIdx.x == 0) init_flag[b] = 0;
}

// One filter's staircase Sigma -> dense row-major N x N (ld = N).
__global__ void k_fused_sym_unpack(const double* __restrict__ s, double* __restrict__ out, int N) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < N * N; e += gridDim.x * blockDim.x) {
        const int r = e / N, c = e - r * N;
        out[e] = s[stair_at(r, c, N)];
    }
}

}  // namespace ekf
