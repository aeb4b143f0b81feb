// Engine 3 ("wide"): a batch of independent filters whose covariances are too large for shared memory (64 < n <= 1,024
// landmarks) and live in HBM, one dense row-major N x ld matrix per filter (the streamed engine's layout, ld = N rounded
// up to 16 doubles).  One launch per SLAM step for the whole batch: a persistent kernel, one filter per CTA at a time,
// strided over the batch.  Per filter and step a CTA runs
//   prediction : k_large_motion's robot block, then k_large_predict_strips (no factors are pending here);
//   first call : every landmark initialised from its reading at the post-prediction pose (k_large_init_landmarks);
//   corrections: for each visible landmark in index order, the arithmetic of k_large_gain_p (the shared helpers of
//                ekf_large_delayed.cuh) at the entry-time pose, appending (K_j, W_j) to the CTA's factor slots;
//   sweep      : once kWidePending factors are pending, and after the last correction, Sigma -= sum_j K_j W_j in one
//                pass through sweep_mma_units<kWidePending> (ekf_large_mma.cuh).  Unused slots of a short group hold
//                zero factors, an exact no-op (fma(-0, 0, v) == v for every v), so one instantiation serves every
//                group size and each element still sees the FMA sequence of one sweep per correction.
// So every filter is bit-identical to an EKF_ENGINE_STREAM filter with carry_pending = 0 fed the same inputs.
#pragma once
#include "ekf_large_mma.cuh"

namespace ekf {

constexpr int kWideMaxN = 1024;  // landmarks: Sigma = 33.9 MB per filter; larger maps are single streamed filters
constexpr int kWidePending = kDefaultPending;
using WideTile = SweepTile<kWidePending>;

struct WideParams {
    double* sigma;                  // [B][N * ld]
    double* state;                  // [B][st_stride]
    int32_t* init_flag;             // [B]
    unsigned long long* n_updates;  // corrections, summed over the batch
    unsigned long long* n_sweeps;   // passes over a filter's Sigma, summed over the batch
    double2* Kp;                    // [grid][kWidePending * ld + 16] factor slots of each CTA
    double2* Wp;
    const double* twists;    // [B][2]
    const double* xy;        // dense: [B][2n]; marker list: [total][2]
    const uint8_t* vis;      // dense: visible flags [B][n]; marker list: ids [total]
    const int32_t* offsets;  // marker list: CSR offsets [B + 1]; null for the dense form
    long long sparse_total;
    long long B;
    long long ld;
    long long slot_stride;  // double2 per CTA in Kp / Wp
    int n, N, st_stride;
    double* nis;  // [B][4] NIS accumulators of k_wide_step<true> (nis() / nis_add())
};

// dynamic shared memory: the sweep's stage ring, then the readings [2n] and visible flags [n] of the current filter
__host__ __device__ inline int wide_smem_bytes(int n) { return WideTile::kSmemBytes + 16 * n + ((n + 15) & ~15); }

__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// One pass over the filter's Sigma with the kWidePending factor slots.  Generic-proxy writes (prediction strips, factor
// slots) are fenced before the bulk copies read them, and the bulk stores are complete before anyone reads Sigma again.
__device__ __forceinline__ void wide_sweep(double* sig, long long ld, int N, const double2* Kp, const double2* Wp,
                                           unsigned char* smem_raw, SweepRing& ring) {
    fence_proxy_async_global();
    __syncthreads();
    sweep_mma_units<kWidePending, false>(sig, ld, N, Kp, Wp, 0, smem_raw, ring);
    if (threadIdx.x == 32 * (kTmaConsumerWarps + 1)) {
        bulk_wait_all();
        fence_proxy_async_global();
    }
    __syncthreads();
}

// NIS: also accumulate the NIS of the step's corrections (none on a filter's first call) into p.nis[b]; thread 0 keeps
// the running sums in shared memory.
template <bool NIS>
__global__ void __launch_bounds__(kTmaThreads, 1) k_wide_step(WideParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* zxy = reinterpret_cast<double*>(smem_raw + WideTile::kSmemBytes);
    uint8_t* zvis = reinterpret_cast<uint8_t*>(zxy + 2 * p.n);
    __shared__ GainSharedP g;
    __shared__ double s_a[2], s_pose[3];
    __shared__ int s_init;
    __shared__ double s_nis[4];
    // per-CTA loop state of the corrections, and the sweep ring's position per role (producer, consumers, storer)
    __shared__ struct {
        int i, pending, dirty;
        unsigned long long corrections, sweeps;
    } L;
    __shared__ int s_ring_stage[3];
    __shared__ uint32_t s_ring_phase[3];
    __shared__ int s_ring_first[3];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int role = warp == 0 ? 0 : (warp <= kTmaConsumerWarps ? 1 : 2);
    if (tid == 0) {
        sweep_mma_init<kWidePending>(smem_raw);
        L.dirty = kWidePending;  // slots >= dirty hold zero factors (the first short group zeroes them all)
        for (int r = 0; r < 3; ++r) {
            s_ring_stage[r] = 0;
            s_ring_phase[r] = 0;
            s_ring_first[r] = 1;
        }
    }
    __syncthreads();
    const int n = p.n, N = p.N;
    const long long ld = p.ld;
    double2* Kp = p.Kp + (long long)blockIdx.x * p.slot_stride;
    double2* Wp = p.Wp + (long long)blockIdx.x * p.slot_stride;

    for (long long b = blockIdx.x; b < p.B; b += gridDim.x) {
        double* sig = p.sigma + b * (long long)N * ld;
        double* st = p.state + b * (long long)p.st_stride;
        // ---- this filter's readings into shared memory; an unlisted marker reads (0, 0) as in the dense arrays
        if (p.offsets) {
            for (int i = tid; i < n; i += kTmaThreads) {
                zxy[2 * i] = 0.0;
                zxy[2 * i + 1] = 0.0;
                zvis[i] = 0;
            }
            __syncthreads();
            const long long begin = p.offsets[b];
            long long count = (long long)p.offsets[b + 1] - begin;
            if (begin < 0 || count < 0 || begin + count > p.sparse_total) count = 0;  // malformed: empty list
            for (long long k = tid; k < count; k += kTmaThreads) {
                const int id = p.vis[begin + k];
                if (id < n) {
                    zxy[2 * id] = p.xy[2 * (begin + k)];
                    zxy[2 * id + 1] = p.xy[2 * (begin + k) + 1];
                    zvis[id] = 1;
                }
            }
        } else {
            for (int i = tid; i < n; i += kTmaThreads) {
                zxy[2 * i] = p.xy[b * 2 * n + 2 * i];
                zxy[2 * i + 1] = p.xy[b * 2 * n + 2 * i + 1];
                zvis[i] = p.vis[b * n + i] != 0;
            }
        }
        // ---- prediction: motion model and robot block (k_large_motion), then the strips (k_large_predict_strips).
        // Sigma is read with ld.global.cg: the sweep's bulk stores bypass L1, so no line of Sigma may live there.
        if (tid == 0) {
            const Motion m = motion_model(st[0], p.twists[2 * b], p.twists[2 * b + 1]);
            double s[3][3];
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) s[r][c] = __ldcg(sig + r * ld + c);
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
            st[0] = st[0] + m.u0;
            st[1] = st[1] + m.u1;
            st[2] = st[2] + m.u2;
            s_a[0] = m.a1;
            s_a[1] = m.a2;
            s_pose[0] = st[0];  // entry-time pose of measurement() (ekf_slam.cpp:109-111)
            s_pose[1] = st[1];
            s_pose[2] = st[2];
            s_init = p.init_flag[b];
        }
        __syncthreads();
        {
            const double a1 = s_a[0], a2 = s_a[1];
            for (int k = 3 + tid; k < N; k += kTmaThreads) {
                const double r0 = __ldcg(sig + k);
                sig[ld + k] = fma(a1, r0, __ldcg(sig + ld + k));
                sig[2 * ld + k] = fma(a2, r0, __ldcg(sig + 2 * ld + k));
                double* row = sig + (long long)k * ld;
                const double c0 = __ldcg(row);
                row[1] = fma(c0, a1, __ldcg(row + 1));
                row[2] = fma(c0, a2, __ldcg(row + 2));
            }
        }
        // ---- first measurement() call: every slot from its reading (k_large_init_landmarks)
        if (!s_init) {
            for (int i = tid; i < n; i += kTmaThreads) {
                double mx, my;
                landmark_from_reading(zxy[2 * i], zxy[2 * i + 1], s_pose[0], s_pose[1], s_pose[2], mx, my);
                st[3 + 2 * i] = mx;
                st[4 + 2 * i] = my;
            }
            if (tid == 0) p.init_flag[b] = 1;
        }
        __syncthreads();
        // ---- corrections in index order; the factors of a group wait in the CTA's slots until the sweep.  The loop
        // state lives in shared memory, so that nothing of it occupies registers during the sweep.
        if (tid == 0) {
            L.i = 0;
            L.pending = 0;
            L.corrections = 0;
            L.sweeps = 0;
            if (NIS) s_nis[0] = s_nis[1] = s_nis[2] = s_nis[3] = 0.0;
        }
        __syncthreads();
        for (;;) {
            int i = L.i;
            while (i < n && !zvis[i]) ++i;  // CTA-uniform
            const bool more = i < n;
            int pending = L.pending;
            const int dirty = L.dirty;
            if (more) {
                const int i3 = 3 + 2 * i;
                if (tid < 5) {
                    const long long ida = tid < 3 ? tid : i3 + (tid - 3);
                    for (int j = 0; j < pending; ++j) g.Kidx[j][tid] = Kp[(long long)j * ld + ida];
                }
                __syncthreads();
                if (warp == 0) {
                    const GainBlockEntry e = gain_block_entry(lane, i3);
                    const Hj h = make_hj(st[i3], st[i3 + 1], s_pose[0], s_pose[1], s_pose[2]);
                    gain_block(lane, e, __ldcg(sig + e.ida * ld + e.idl), Wp, ld, pending, h, zxy[2 * i], zxy[2 * i + 1],
                               g);
                }
                __syncthreads();
                if (NIS && tid == 0 && s_init) nis_add(s_nis, nis(g.si, g.nu0, g.nu1));
                double2* Kout = Kp + (long long)pending * ld;
                double2* Wout = Wp + (long long)pending * ld;
                const long long i3l = (long long)i3 * ld;
                for (long long k = tid; k < ld; k += kTmaThreads) {
                    double2 wk = make_double2(0.0, 0.0), kk = make_double2(0.0, 0.0);  // padding columns: zero factor
                    if (k < N) {
                        double s0 = __ldcg(sig + k), s1 = __ldcg(sig + ld + k), s2 = __ldcg(sig + 2 * ld + k),
                               s3 = __ldcg(sig + i3l + k), s4 = __ldcg(sig + i3l + ld + k);
                        gain_rows_rebuild(s0, s1, s2, s3, s4, Wp, ld, k, pending, g);
                        st[k] = gain_column(g, s0, s1, s2, s3, s4, st[k], k, wk, kk);
                    }
                    Wout[k] = wk;
                    Kout[k] = kk;
                }
                ++pending;
            }
            const bool flush = pending == kWidePending || (!more && pending > 0);
            if (flush && pending < kWidePending) {
                // short group: the slots pending .. dirty-1 still hold factors of an earlier group
                for (long long e = tid; e < (long long)(dirty - pending) * ld; e += kTmaThreads) {
                    Kp[(long long)pending * ld + e] = make_double2(0.0, 0.0);
                    Wp[(long long)pending * ld + e] = make_double2(0.0, 0.0);
                }
            }
            __syncthreads();  // everyone has read L
            if (tid == 0) {
                L.i = i + 1;
                L.pending = flush ? 0 : pending;
                L.dirty = flush && pending < kWidePending ? pending : (pending > dirty ? pending : dirty);
                L.corrections += more ? 1 : 0;
                L.sweeps += flush ? 1 : 0;
            }
            if (flush) {
                SweepRing ring;
                ring.stage = s_ring_stage[role];
                ring.phase = s_ring_phase[role];
                ring.first = s_ring_first[role] != 0;
                wide_sweep(sig, ld, N, Kp, Wp, smem_raw, ring);
                if (lane == 0 && (warp == 0 || warp == 1 || warp == kTmaConsumerWarps + 1)) {
                    s_ring_stage[role] = ring.stage;
                    s_ring_phase[role] = ring.phase;
                    s_ring_first[role] = ring.first ? 1 : 0;
                }
            }
            __syncthreads();
            if (!more) break;
        }
        if (tid == 0 && L.corrections) {
            atomicAdd(p.n_updates, L.corrections);
            atomicAdd(p.n_sweeps, L.sweeps);
            if (NIS) {
                for (int k = 0; k < 4; ++k) p.nis[4 * b + k] += s_nis[k];
            }
        }
        __syncthreads();  // zxy / zvis are refilled for the next filter
    }
    if (threadIdx.x == 32 * (kTmaConsumerWarps + 1)) bulk_wait_all();
}

// One step of the whole batch on `device`.  grid = the number of CTAs the factor slots were allocated for.
template <bool NIS>
inline cudaError_t launch_wide_step(const WideParams& p, int grid, cudaStream_t stream, int device) {
    const cudaError_t e = kernel_setup<k_wide_step<NIS>>(device, kTmaThreads, wide_smem_bytes(kWideMaxN), false);
    if (e != cudaSuccess) return e;
    k_wide_step<NIS><<<(unsigned)grid, kTmaThreads, wide_smem_bytes(p.n), stream>>>(p);
    return cudaGetLastError();
}

}  // namespace ekf
