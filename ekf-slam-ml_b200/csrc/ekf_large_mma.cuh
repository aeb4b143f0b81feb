// Multi-factor covariance sweep of the streamed engine on the FP64 tensor-core path.
//
// One sweep applies the P pending corrections, Sigma <- Sigma - sum_{j<P} K_j W_j (ekf_large_delayed.cuh), i.e. a
// rank-2P update: per 8 x 8 block of Sigma a product [-K_0 .. -K_{P-1}] (8 x 2P) times [W_0 ; .. ; W_{P-1}] (2P x 8),
// which mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4) does in ceil(2P / 4) instructions.  DMMA accumulates its k = 0..3 terms
// as a chain of FMAs in order (experiments/dmma_rate.cu), and the k axis is laid out factor by factor, x before y, so
// every element still sees exactly the FMA sequence of sequential sweeps: the result is bit-identical to
// k_large_sweep_p (tests/test_gpu_ekf.py::test_delayed_application_is_bit_identical).
//
// What DMMA changes is the instruction mix.  Vector consumers issue 2P DFMA per element plus one shared-memory K fetch
// per four of them, which at P = 14 pushed the sweep from the copy time (0.66 ms at N = 16,387) to 0.85 ms.  Here a
// warp issues ceil(P/2) DMMA per 64 elements; its B fragments (the W pairs of its columns) sit in registers for the
// whole work unit and the A fragments (the stage's K rows) cost ceil(P/2) 8-byte loads per 8 rows.  The FP64 pipe time
// is the same as for the vector form (both run at 64 FMA / clk / SM), but it is the ONLY cost left next to the copy,
// and it stays below the copy time up to P ~ 22.
//
// CTA = 1 producer warp + 8 consumer warps + 1 store warp, one CTA per SM, persistent over work units of SweepTile<P>
// columns x kUnitRows rows, moved by the bulk copy engine (cp.async.bulk, SASS UBLKCP) through a ring of mbarrier
// stages:
//   producer : waits empty[s], bulk-loads the stage's row segments and its K rows (P x SROWS pairs); full[s] counts bytes;
//   consumers: wait full[s], run the DMMA blocks of their columns in place in shared memory, arrive on done[s];
//   storer   : waits done[s], bulk-stores the row segments, and hands stage s-1 back (empty[s-1]) once the store of
//              s-1 has finished reading shared memory.
// Stage rows are padded by 8 doubles so that the fragment accesses (lane (g, t) touches row g, columns 2t, 2t+1 of a
// block) are bank-conflict free.
#pragma once
#include "bulk_copy.cuh"
#include "ekf_large_delayed.cuh"
#include "host_util.cuh"

namespace ekf {

constexpr int kUnitRows = 128;  // rows of a work unit
constexpr int kTmaConsumerWarps = 8;
constexpr int kTmaThreads = 32 * (kTmaConsumerWarps + 2);

// The sweep's geometry, from P alone.  A consumer warp keeps NBW x ceil(P/2) W fragment doubles in registers: at 64
// columns per warp that fits up to P = 14, so deeper groups get 256-column tiles (32 columns per warp) with 16-row
// stages, which keeps a stage at ~33 KB.  Measured on B200 (experiments/README.md): 6 stages slower, 256 columns 8 %
// slower at P = 14, unguarded DMMA blocks slower.
template <int P>
struct SweepTile {
    static constexpr int COLS = P <= 14 ? 512 : 256;  // tile width
    static constexpr int SROWS = P <= 14 ? 8 : 16;    // rows per stage
    static constexpr int STAGES = 4;
    static constexpr int KS = (2 * P + 3) / 4;                  // DMMA k-steps
    static constexpr int NBW = COLS / (8 * kTmaConsumerWarps);  // 8 x 8 blocks per consumer warp and 8 rows
    static constexpr int RG = SROWS / 8;                        // 8-row groups per stage
    static constexpr int RS = COLS + 8;  // row stride in doubles: 64 B past a multiple of 128 B
    static constexpr int kTileBytes = SROWS * RS * 8;
    static constexpr int kKBytes = P * SROWS * 16;
    static constexpr int kSmemBytes = STAGES * (kTileBytes + kKBytes) + 3 * STAGES * 8 + 64;
};

// Where one thread stands in the CTA's stage ring: each role (producer lane, consumer warps, store lane) advances its own
// copy.  A kernel that sweeps several times keeps it across calls, so the ring runs on as one stream of stages.
struct SweepRing {
    int stage = 0;
    uint32_t phase = 0;
    bool first = true;  // store lane: no earlier stage to hand back yet
};

// The barriers of the stage ring in the dynamic shared memory `smem_raw` (laid out as SweepTile<P>); every thread of the
// CTA must pass a __syncthreads() before the first sweep.
template <int P>
__device__ __forceinline__ uint64_t* sweep_mma_barriers(unsigned char* smem_raw) {
    using T = SweepTile<P>;
    return reinterpret_cast<uint64_t*>(smem_raw + (size_t)T::STAGES * (T::kTileBytes + T::kKBytes));
}
template <int P>
__device__ __forceinline__ void sweep_mma_init(unsigned char* smem_raw) {
    uint64_t* full = sweep_mma_barriers<P>(smem_raw);
    for (int s = 0; s < SweepTile<P>::STAGES; ++s) {
        mbar_init(full + s, 1);
        mbar_init(full + SweepTile<P>::STAGES + s, kTmaConsumerWarps);
        mbar_init(full + 2 * SweepTile<P>::STAGES + s, 1);
    }
    fence_mbar_init();
}

// The work units of one sweep, run by all kTmaThreads threads of the CTA: blockIdx.x, blockIdx.x + gridDim.x, ... when
// the grid shares the sweep (GRID), all of them otherwise.  The bulk stores of the last stages may still be in flight
// on return: the store lane drains them (bulk_wait_all) before anything reads the swept rows or the CTA exits.
template <int P, bool GRID>
__device__ __forceinline__ void sweep_mma_units(double* sig, long long ld, int n_rows, const double2* Kp, const double2* Wp,
                                                long long row0, unsigned char* smem_raw, SweepRing& ring) {
    using T = SweepTile<P>;
    constexpr int COLS = T::COLS, SROWS = T::SROWS, STAGES = T::STAGES, KS = T::KS, NBW = T::NBW, RG = T::RG,
                  RS = T::RS;
    double* tiles = reinterpret_cast<double*>(smem_raw);                                   // [STAGES][SROWS][RS]
    double2* ksm = reinterpret_cast<double2*>(smem_raw + (size_t)STAGES * T::kTileBytes);  // [STAGES][P][SROWS]
    uint64_t* full = sweep_mma_barriers<P>(smem_raw);
    uint64_t* done = full + STAGES;
    uint64_t* empty = done + STAGES;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    const int chunks = (int)((ld + COLS - 1) / COLS);
    const int row_units = (n_rows + kUnitRows - 1) / kUnitRows;
    const long long units = (long long)chunks * row_units;
    int stage = ring.stage;
    uint32_t phase = ring.phase;
    bool first = ring.first;

    for (long long u = GRID ? blockIdx.x : 0; u < units; u += GRID ? gridDim.x : 1) {
        const int cu = (int)(u % chunks), ru = (int)(u / chunks);
        const long long c0 = (long long)cu * COLS;
        const int width = (int)(ld - c0 < COLS ? ld - c0 : COLS);  // multiple of 16 doubles
        const int r_begin = ru * kUnitRows;
        const int r_end = r_begin + kUnitRows < n_rows ? r_begin + kUnitRows : n_rows;
        const int groups = (r_end - r_begin + SROWS - 1) / SROWS;
        if (warp == 0) {
            // ---------------------------------------------------------------- producer
            if (lane == 0) {
                for (int g = 0; g < groups; ++g) {
                    mbar_wait(empty + stage, phase ^ 1u);
                    const int r = r_begin + g * SROWS;
                    const int nr = r_end - r < SROWS ? r_end - r : SROWS;
                    mbar_arrive_expect_tx(full + stage, (uint32_t)(nr * width * 8 + P * SROWS * 16));
                    double* tile = tiles + (size_t)stage * SROWS * RS;
                    for (int k = 0; k < nr; ++k)
                        bulk_g2s(tile + k * RS, sig + (long long)(r + k) * ld + c0, (uint32_t)(width * 8), full + stage);
                    for (int j = 0; j < P; ++j)
                        bulk_g2s(ksm + ((size_t)stage * P + j) * SROWS, Kp + (long long)j * ld + row0 + r, SROWS * 16, full + stage);
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        } else if (warp <= kTmaConsumerWarps) {
            // ---------------------------------------------------------------- consumers
            const int w = warp - 1;
            const int g = lane >> 2, t = lane & 3;
            const int wc0 = 8 * NBW * w;  // this warp's first column inside the tile
            // B fragments: B[k][n] of k-step s and block b = W_j[c0 + wc0 + 8 b + g].{x | y}, j = (4 s + t) / 2,
            // component (4 s + t) % 2; zero beyond the last factor or the tile's width
            double bf[NBW][KS];
#pragma unroll
            for (int b = 0; b < NBW; ++b) {
                const int c = wc0 + 8 * b + g;
#pragma unroll
                for (int s = 0; s < KS; ++s) {
                    const int kk = 4 * s + t, j = kk >> 1;
                    bf[b][s] = (j < P && c < width)
                                   ? reinterpret_cast<const double*>(Wp + (long long)j * ld + c0 + c)[kk & 1]
                                   : 0.0;
                }
            }
            const int nblk = width - wc0 >= 8 * NBW ? NBW : (width - wc0 > 0 ? (width - wc0) / 8 : 0);  // warp-uniform
            for (int gi = 0; gi < groups; ++gi) {
                mbar_wait(full + stage, phase);
                double* tile = tiles + (size_t)stage * SROWS * RS;
                const double* kst = reinterpret_cast<const double*>(ksm + (size_t)stage * P * SROWS);
#pragma unroll
                for (int rg = 0; rg < RG; ++rg) {
                    double af[KS];  // A[g][k] = -K_j[row 8 rg + g of the stage].{x | y}
#pragma unroll
                    for (int s = 0; s < KS; ++s) {
                        const int kk = 4 * s + t, j = kk >> 1;
                        af[s] = j < P ? -kst[2 * (j * SROWS + 8 * rg + g) + (kk & 1)] : 0.0;
                    }
                    double* cp = tile + (8 * rg + g) * RS + wc0 + 2 * t;
                    double2 cf[NBW];
#pragma unroll
                    for (int b = 0; b < NBW; ++b)
                        if (b < nblk) cf[b] = *reinterpret_cast<const double2*>(cp + 8 * b);
#pragma unroll
                    for (int s = 0; s < KS; ++s)
#pragma unroll
                        for (int b = 0; b < NBW; ++b)
                            if (b < nblk)
                                asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                                             : "+d"(cf[b].x), "+d"(cf[b].y)
                                             : "d"(af[s]), "d"(bf[b][s]));
#pragma unroll
                    for (int b = 0; b < NBW; ++b)
                        if (b < nblk) *reinterpret_cast<double2*>(cp + 8 * b) = cf[b];
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(done + stage);
                if (++stage == STAGES) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
        } else {
            // ---------------------------------------------------------------- store warp
            if (lane == 0) {
                for (int g = 0; g < groups; ++g) {
                    const int r = r_begin + g * SROWS;
                    const int nr = r_end - r < SROWS ? r_end - r : SROWS;
                    mbar_wait(done + stage, phase);
                    double* tile = tiles + (size_t)stage * SROWS * RS;
                    for (int k = 0; k < nr; ++k)
                        bulk_s2g(sig + (long long)(r + k) * ld + c0, tile + k * RS, (uint32_t)(width * 8));
                    bulk_commit();
                    bulk_wait_read_1();  // every store but the newest has finished reading shared memory
                    if (!first) mbar_arrive(empty + (stage == 0 ? STAGES - 1 : stage - 1));
                    first = false;
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
    }
    ring.stage = stage;
    ring.phase = phase;
    ring.first = first;
}

template <int P>
__global__ void __launch_bounds__(kTmaThreads, 1)
    k_large_sweep_mma(double* __restrict__ sig, long long ld, int n_rows, const double2* __restrict__ Kp,
                      const double2* __restrict__ Wp, long long row0, unsigned long long* __restrict__ n_updates,
                      int n_counted, const UpdateCmd* __restrict__ cmd) {
    pdl_prologue();
    if (cmd && !cmd->do_update) return;
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_updates) *n_updates += (unsigned long long)n_counted;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    if (threadIdx.x == 0) sweep_mma_init<P>(smem_raw);
    __syncthreads();
    SweepRing ring;
    sweep_mma_units<P, true>(sig, ld, n_rows, Kp, Wp, row0, smem_raw, ring);
    if (threadIdx.x == 32 * (kTmaConsumerWarps + 1)) bulk_wait_all();  // drain before the CTA's shared memory goes away
}

// One persistent CTA per SM (at most one per work unit).  P is at most kMaxPending: the factor buffers have no more
// slots, and -DEKF_MAX_PENDING=14 builds no deeper kernel.
template <int P>
cudaError_t launch_sweep_mma(double* sig, long long ld, int n_rows, const double2* Kp, const double2* Wp, long long row0,
                             unsigned long long* n_updates, int n_counted, const UpdateCmd* cmd, int sm_count,
                             cudaStream_t stream) {
    if constexpr (P > kMaxPending) {
        return cudaErrorInvalidValue;
    } else {
        using T = SweepTile<P>;
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess) dev = -1;
        const cudaError_t e = kernel_setup<k_large_sweep_mma<P>>(dev, kTmaThreads, T::kSmemBytes, false);
        if (e != cudaSuccess) return e;
        const long long units = ((ld + T::COLS - 1) / T::COLS) * ((n_rows + kUnitRows - 1) / kUnitRows);
        const unsigned grid = (unsigned)(units < sm_count ? (units < 1 ? 1 : units) : sm_count);
        k_large_sweep_mma<P><<<grid, kTmaThreads, T::kSmemBytes, stream>>>(sig, ld, n_rows, Kp, Wp, row0, n_updates,
                                                                          n_counted, cmd);
        return cudaGetLastError();
    }
}

// Apply `pending` factor pairs: the register path for 1-2 factors, the DMMA pipeline from 3 on.  Kp must have at least
// 16 pairs of slack after its last used row (a stage's K rows are fetched SweepTile<P>::SROWS at a time).
inline cudaError_t launch_sweep(int pending, double* sig, long long ld, int n_rows, const double2* Kp, const double2* Wp,
                                long long row0, unsigned long long* n_updates, int n_counted, const UpdateCmd* cmd,
                                int sm_count, cudaStream_t stream) {
    switch (pending) {
        case 1:
        case 2: return launch_sweep_p(pending, sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, stream);
        case 3: return launch_sweep_mma<3>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 4: return launch_sweep_mma<4>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 5: return launch_sweep_mma<5>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 6: return launch_sweep_mma<6>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 7: return launch_sweep_mma<7>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 8: return launch_sweep_mma<8>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 9: return launch_sweep_mma<9>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 10: return launch_sweep_mma<10>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 11: return launch_sweep_mma<11>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 12: return launch_sweep_mma<12>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 13: return launch_sweep_mma<13>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 14: return launch_sweep_mma<14>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 15: return launch_sweep_mma<15>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 16: return launch_sweep_mma<16>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 17: return launch_sweep_mma<17>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 18: return launch_sweep_mma<18>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 19: return launch_sweep_mma<19>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        case 20: return launch_sweep_mma<20>(sig, ld, n_rows, Kp, Wp, row0, n_updates, n_counted, cmd, sm_count, stream);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace ekf
