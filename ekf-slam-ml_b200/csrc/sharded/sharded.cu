// Engine 3: one filter, covariance row-block-sharded over `world` GPUs (include/ekf_sharded_b200.h).
// The O(N^2) sweep and the O(N) gathers run on each rank's own rows.  Per correction the ranks exchange W = Hj Sigma:
// the row owners' partial products are pushed into every rank's buffer over NVLink (k_sh_correct_push) or summed by an
// NCCL all-reduce; every rank then forms all of K and the state update itself.  A single-process "local" mode keeps
// `world` shards on one device and replaces the NCCL calls by device copies, so that the sharding arithmetic can be
// parity-tested on one GPU.  Motion, association and gain arithmetic are the streamed engine's (ekf_large*.cuh).
// Restates rigid2d/src/ekf_slam.cpp:55-106, 108-197, 200-214, 217-276, 278-402.
#include <cuda_runtime.h>
#include <nccl.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "../../../include/ekf_sharded_b200.h"
#include "../ekf_large_mma.cuh"
#include "../host_util.cuh"

using namespace ekf;

namespace {

#define NC(expr)                                                                               \
    do {                                                                                       \
        ncclResult_t r_ = (expr);                                                              \
        if (r_ != ncclSuccess) return fail(1000 + (int)r_, "%s failed: %s (line %d)", #expr, ncclGetErrorString(r_), __LINE__); \
    } while (0)

// per-correction scalars, replicated on every shard
struct Ctx {
    Hj h;
    double sx, sy;
    int i3, active;
};

// ---- prediction (the motion model and the robot block: k_large_motion on every shard)
__global__ void k_sh_predict_rows12(double* __restrict__ sig, long long ld, int N, const double* __restrict__ motion) {
    const int k = 3 + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    const double r0 = sig[k];
    sig[ld + k] = fma(motion[0], r0, sig[ld + k]);
    sig[2 * ld + k] = fma(motion[1], r0, sig[2 * ld + k]);
}
// local rows [lr_begin, rows): columns 1,2 += a * column 0
__global__ void k_sh_predict_cols(double* __restrict__ sig_local, long long ld, int lr_begin, int rows,
                                  const double* __restrict__ motion) {
    const int lr = lr_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (lr >= rows) return;
    double* row = sig_local + (long long)lr * ld;
    const double c0 = row[0];
    row[1] = fma(c0, motion[0], row[1]);
    row[2] = fma(c0, motion[1], row[2]);
}

// ---- correction
__global__ void k_sh_ctx_h(const double* __restrict__ state, const double* __restrict__ pose_src,
                           const UpdateCmd* __restrict__ cmd, int lm_arg, double sx_arg, double sy_arg,
                           Ctx* __restrict__ ctx) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int lm = lm_arg, active = 1;
    double sx = sx_arg, sy = sy_arg;
    if (cmd) {
        active = cmd->do_update;
        lm = cmd->lm;
        sx = cmd->sx;
        sy = cmd->sy;
    }
    ctx->active = active;
    if (!active) return;
    const int i3 = 3 + 2 * lm;
    ctx->i3 = i3;
    ctx->h = make_hj(state[i3], state[i3 + 1], pose_src[0], pose_src[1], pose_src[2]);
    ctx->sx = sx;
    ctx->sy = sy;
}

// partial W = Hj * Sigma_current restricted to the rows this shard owns (zeros stand in for the others).
// Sigma_current = Sigma_0 - sum_{j<p} K_j W_j is rebuilt on the fly from the pending factors (ekf_large_delayed.cuh).
__global__ void __launch_bounds__(256)
    k_sh_wpart(const double* __restrict__ sig_local, long long ld, long long r0, long long r1, int N,
               const Ctx* __restrict__ ctx, const double2* __restrict__ Kp, const double2* __restrict__ Wp, int p,
               double2* __restrict__ Wpart) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ld) return;
    double2 w = make_double2(0.0, 0.0);
    if (c < N && ctx->active) {
        const long long id[5] = {0, 1, 2, ctx->i3, ctx->i3 + 1};
        double s[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            double v = 0.0;
            if (id[k] >= r0 && id[k] < r1) {
                v = sig_local[(id[k] - r0) * ld + c];
                for (int j = 0; j < p; ++j) v = apply_factor(v, Kp[(long long)j * ld + id[k]], Wp[(long long)j * ld + c]);
            }
            s[k] = v;
        }
        const Hj h = ctx->h;
        w = make_double2(h_row0(h, s[1], s[2], s[3], s[4]), h_row1(h, s[0], s[1], s[2], s[3], s[4]));
    }
    Wpart[c] = w;  // a dropped measurement contributes a zero factor
}

// After the all-reduce every rank holds the full W = Hj Sigma.  With Sigma symmetric (kept to rounding by the
// reference's (I - K H) Sigma, SURVEY.md §8e) K = Sigma Hj^T S^-1 = W^T S^-1, so every replica forms ALL of K and the
// state update locally: no strided column reads of the local rows and no exchange of K.
__global__ void __launch_bounds__(256)
    k_sh_gain_state(const double2* __restrict__ Wp_slot, double2* __restrict__ Kout, double* __restrict__ state,
                    const Ctx* __restrict__ ctx, int N, long long ld) {
    __shared__ Sym2 si_s;
    __shared__ double nu_s[2];
    __shared__ int active_s;
    if (threadIdx.x == 0) {
        active_s = ctx->active;
        if (active_s) {
            const int i3 = ctx->i3;
            const double2 w5[5] = {Wp_slot[0], Wp_slot[1], Wp_slot[2], Wp_slot[i3], Wp_slot[i3 + 1]};
            gain_scalars(ctx->h, w5, ctx->sx, ctx->sy, ref_noise(), si_s, nu_s[0], nu_s[1]);
        }
    }
    __syncthreads();
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= ld) return;
    if (k >= N || !active_s) {
        Kout[k] = make_double2(0.0, 0.0);
        return;
    }
    double2 kk;
    state[k] = gain_state(si_s, nu_s[0], nu_s[1], Wp_slot[k], state[k], k, kk);
    Kout[k] = kk;
}

// ---- the W exchange without a collective ("push") ----------------------------------------------------------------
// Only two ranks hold rows that enter W = Hj Sigma: rank 0 (robot rows 0..2) and the owner of landmark i.  Instead of
// an all-reduce of a 2 ld vector of which at most two contributions are non-zero, those two ranks store their partial
// W straight into every rank's exchange buffer over NVLink - through the NVSwitch multicast address when there is one
// (one store, replicated by the switch), else peer by peer - and raise a flag; every rank then adds the two partials
// inside the gain kernel, which waits on the flags instead of on a collective.
// Exchange buffer per rank (symmetric, allocated by the caller, see ekf_sharded_attach_exchange):
//   flags [kMaxPending][2][256-column blocks] uint64 (pad to 256 B) | data [kMaxPending][2][ld] double2
// Slot p = the pending-factor slot of the correction, source 0 = rank 0's partial, source 1 = the landmark owner's.  A flag
// holds the group generation number of the data it guards; slots are reused only after the group's sweep, which is
// preceded by a barrier across the ranks.
__host__ __device__ inline size_t xflag_blocks(long long ld) { return (size_t)((ld + 255) / 256); }
__host__ __device__ inline size_t xflag_bytes(long long ld) {
    return ((size_t)kMaxPending * 2 * xflag_blocks(ld) * sizeof(unsigned long long) + 255) & ~(size_t)255;
}
__host__ __device__ inline size_t xdata_index(int p, int src, long long ld) { return ((size_t)p * 2 + src) * (size_t)ld; }

__device__ __forceinline__ void st_sys_v2(double2* ptr, double2 v) {  // also valid on a multicast address
    asm volatile("st.relaxed.sys.global.v2.f64 [%0], {%1, %2};" ::"l"(ptr), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void mc_st_v2(double2* ptr, double2 v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(ptr),
                 "r"(__double2loint(v.x)), "r"(__double2hiint(v.x)), "r"(__double2loint(v.y)), "r"(__double2hiint(v.y))
                 : "memory");
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* ptr, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(ptr), "l"(v) : "memory");
}
__device__ __forceinline__ void mc_st_release_u64(unsigned long long* ptr, unsigned long long v) {
    asm volatile("fence.acq_rel.sys;" ::: "memory");
    asm volatile("multimem.st.relaxed.sys.global.u64 [%0], %1;" ::"l"(ptr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* ptr) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(ptr) : "memory");
    return v;
}

struct XPeers {
    unsigned char* base[8];  // every rank's exchange buffer as mapped here (index = rank)
    unsigned char* mc;       // multicast address of the same buffer, or null
    int world;
};

#ifndef EKF_SH_PROF
#define EKF_SH_PROF 0  // 1: per-phase globaltimer stamps of the fused correction kernel (development builds only)
#endif
#if EKF_SH_PROF
__device__ unsigned long long g_sh_prof[2][8];
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define SH_MARK(k)                                                                  \
    do {                                                                            \
        if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))   \
            g_sh_prof[blockIdx.x == 0 ? 0 : 1][k] = gtime();                        \
    } while (0)
#else
#define SH_MARK(k) \
    do {           \
    } while (0)
#endif

// The whole correction in ONE launch.  Per 256-column block b of a rank:
//   source ranks (rank 0: rows 0..2; the landmark's owner: rows 3+2i, 4+2i): rebuild the owned rows' column entries
//   with the pending factors, form the partial W, store it into every rank's slot and raise the block's flag;
//   every rank: wait for the flags of block b and of the blocks holding columns {0,1,2,3+2i,4+2i} (they carry S),
//   then W = sum of the partials, S^-1, K, the state update and the factor slot for the sweep.
// A CTA pushes before it waits and waits only on pushes, and with programmatic stream serialisation a successor's CTAs
// are admitted only after every CTA of this grid has started, so all flags a CTA waits for are eventually raised.
// That needs the whole grid resident at once, which ekf_sharded_attach_exchange checks.
// Measured (2 GPUs, N = 80,003): ~2.5 us pose/landmark/H_j and row loads, ~2 us partial W + stores, ~10 us until the
// 1.3 MB of partials are visible on the peers (the release fence waits for the multicast acknowledgements; sending
// self-validating lines instead of data + flag moved twice the bytes in the same time), ~1 us S^-1.
__global__ void __launch_bounds__(256)
    k_sh_correct_push(const double* __restrict__ sig_local, long long ld, long long r0, long long r1, long long r1_rank0, int N,
                      int rank, double* __restrict__ state, const double* __restrict__ pose_src,
                      const UpdateCmd* __restrict__ cmd, int lm_arg, double sx_arg, double sy_arg, double2* __restrict__ Kall,
                      double2* __restrict__ Wall, int p, const XPeers xp, const unsigned char* __restrict__ xlocal,
                      unsigned long long gen, unsigned long long* __restrict__ read_count, unsigned long long read_target) {
    __shared__ Hj h_s;
    __shared__ double z_s[2], nu_s[2];
    __shared__ Sym2 si_s;
    __shared__ double2 kidx_s[kMaxPending][5];
    SH_MARK(0);
    pdl_prologue();
    SH_MARK(1);
    int lm = lm_arg, active = 1;
    double sx = sx_arg, sy = sy_arg;
    if (cmd) {
        active = cmd->do_update;
        lm = cmd->lm;
        sx = cmd->sx;
        sy = cmd->sy;
    }
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double2* Wslot = Wall + (long long)p * ld;
    double2* Kout = Kall + (long long)p * ld;
    if (!active) {  // a dropped measurement: every rank knows (the command block is replicated), nothing is exchanged
        if (threadIdx.x == 0) atomicAdd(read_count, 1ull);
        if (c < ld) {
            Wslot[c] = make_double2(0.0, 0.0);
            Kout[c] = make_double2(0.0, 0.0);
        }
        return;
    }
    const long long i3 = 3 + 2 * (long long)lm;
    const bool two_sources = i3 >= r1_rank0;  // the landmark's rows are not rank 0's
    const bool owns_lm = i3 >= r0 && i3 < r1;
    const bool source = rank == 0 || owns_lm;
    const int my_src = rank == 0 ? 0 : 1;
    const long long id[5] = {0, 1, 2, i3, i3 + 1};
    const size_t nblk = xflag_blocks(ld);
    // Thread 0 of every CTA reads the pose and the landmark from the state that other CTAs update at the end of this
    // same kernel: it counts itself in once it has them, and the (at most three) CTAs that own those elements hold
    // their state update back until every CTA of the grid has counted in.
    if (threadIdx.x == 0) {
        const double lx = state[i3], ly = state[i3 + 1], p0 = pose_src[0], p1 = pose_src[1], p2 = pose_src[2];
        h_s = make_hj(lx, ly, p0, p1, p2);
        __threadfence();
        atomicAdd(read_count, 1ull);
        z_s[0] = sx;
        z_s[1] = sy;
    }
    double sv[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    bool own[5] = {false, false, false, false, false};
    if (source) {
        if (threadIdx.x >= 32 && threadIdx.x < 37) {
            const int k = threadIdx.x - 32;
            if (id[k] >= r0 && id[k] < r1)
                for (int j = 0; j < p; ++j) kidx_s[j][k] = Kall[(long long)j * ld + id[k]];
        }
        if (c < N) {
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                own[k] = id[k] >= r0 && id[k] < r1;
                sv[k] = own[k] ? sig_local[(id[k] - r0) * ld + c] : 0.0;
            }
        }
    }
    __syncthreads();
    SH_MARK(2);
    if (source) {
        if (c < ld) {
            double2 w = make_double2(0.0, 0.0);
            if (c < N) {
#pragma unroll 4
                for (int j = 0; j < p; ++j) {
                    const double2 wj = Wall[(long long)j * ld + c];
#pragma unroll
                    for (int k = 0; k < 5; ++k)
                        if (own[k]) sv[k] = apply_factor(sv[k], kidx_s[j][k], wj);
                }
                const Hj h = h_s;
                w = make_double2(h_row0(h, sv[1], sv[2], sv[3], sv[4]), h_row1(h, sv[0], sv[1], sv[2], sv[3], sv[4]));
            }
            const size_t o = xflag_bytes(ld) + (xdata_index(p, my_src, ld) + (size_t)c) * sizeof(double2);
            if (xp.mc) {
                mc_st_v2(reinterpret_cast<double2*>(xp.mc + o), w);
            } else {
                for (int g = 0; g < xp.world; ++g) st_sys_v2(reinterpret_cast<double2*>(xp.base[g] + o), w);
            }
        }
        SH_MARK(3);
        // the CTA's stores happen before the barrier; thread 0's system-scope fence after it (inside the release
        // below) is cumulative over them, so one fence per CTA orders the whole block's partial before its flag
        __syncthreads();
        if (threadIdx.x == 0) {
            const size_t of = (((size_t)p * 2 + my_src) * nblk + blockIdx.x) * sizeof(unsigned long long);
            if (xp.mc) {
                mc_st_release_u64(reinterpret_cast<unsigned long long*>(xp.mc + of), gen);
            } else {
                for (int g = 0; g < xp.world; ++g)
                    st_release_sys_u64(reinterpret_cast<unsigned long long*>(xp.base[g] + of), gen);
            }
        }
        SH_MARK(4);
    }
    // ---- every rank: the partials of this block and of the blocks that carry S
    if (threadIdx.x < 8) {
        const int src = threadIdx.x & 1, which = threadIdx.x >> 1;
        if (src == 0 || two_sources) {
            const size_t blk = which == 0 ? (size_t)blockIdx.x : which == 1 ? 0 : (size_t)((i3 + (which - 2)) >> 8);
            const unsigned long long* fl = reinterpret_cast<const unsigned long long*>(xlocal) + ((size_t)p * 2 + src) * nblk + blk;
            while (ld_acquire_sys_u64(fl) != gen) {
            }
        }
    }
    __syncthreads();
    SH_MARK(6);
    const double2* x0 = reinterpret_cast<const double2*>(xlocal + xflag_bytes(ld)) + xdata_index(p, 0, ld);
    const double2* x1 = reinterpret_cast<const double2*>(xlocal + xflag_bytes(ld)) + xdata_index(p, 1, ld);
    if (threadIdx.x == 0) {
        const Hj h = h_s;
        double2 w5[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            w5[k] = __ldcg(x0 + id[k]);
            if (two_sources) {
                const double2 b = __ldcg(x1 + id[k]);
                w5[k] = make_double2(w5[k].x + b.x, w5[k].y + b.y);
            }
        }
        gain_scalars(h, w5, z_s[0], z_s[1], ref_noise(), si_s, nu_s[0], nu_s[1]);
        const long long b0 = (long long)blockIdx.x << 8, b1 = b0 + 256;
        if (b0 < 3 || (i3 + 1 >= b0 && i3 < b1)) {  // this CTA's state update overwrites what thread 0 of the others reads
            while (ld_acquire_sys_u64(read_count) < read_target) {
            }
        }
    }
    __syncthreads();
    SH_MARK(7);
    if (c >= ld) return;
    if (c >= N) {
        Wslot[c] = make_double2(0.0, 0.0);
        Kout[c] = make_double2(0.0, 0.0);
        return;
    }
    double2 w = __ldcg(x0 + c);
    if (two_sources) {
        const double2 b = __ldcg(x1 + c);
        w = make_double2(w.x + b.x, w.y + b.y);
    }
    Wslot[c] = w;
    double2 kk;
    state[c] = gain_state(si_s, nu_s[0], nu_s[1], w, state[c], c, kk);
    Kout[c] = kk;
}

// ---- association
// this shard's landmarks [L0, L1): the shard's minimum and runner-up, merged later in rank order by k_sh_decide
__global__ void __launch_bounds__(256)
    k_sh_assoc_local(const double* __restrict__ robot, const double* __restrict__ sig_local, long long ld, long long r0,
                     int L0, int L1, const double* __restrict__ state, const double* __restrict__ meas, int j,
                     const int* __restrict__ known_count_p, AssocPartial* __restrict__ block_partials,
                     unsigned int* __restrict__ done_counter, AssocPartial* __restrict__ out) {
    const int known_count = *known_count_p;
    double zr, zphi;
    range_bearing(meas[2 * j], meas[2 * j + 1], zr, zphi);
    double best, second;
    int best_i;
    if (assoc_scan(robot, sig_local, ld, r0, L0, L1 < known_count ? L1 : known_count, state, zr, zphi, state[0],
                   state[1], state[2], block_partials, done_counter, best, second, best_i, ref_noise()))
        *out = AssocPartial{best, second, best_i, 0};
}

// identical on every replica: merge the per-rank partials in rank order and take the decision
__global__ void k_sh_decide(const AssocPartial* __restrict__ parts, int world, double* __restrict__ state, int n,
                            const double* __restrict__ meas, int j, int* __restrict__ known_count_p,
                            UpdateCmd* __restrict__ cmd, int32_t* __restrict__ assoc_out, double* __restrict__ dmin_out,
                            double* __restrict__ second_out, uint8_t* __restrict__ created_out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double best = INFINITY, second = INFINITY;
    int best_i = 0x7fffffff;
    for (int g = 0; g < world; ++g) assoc_merge(best, second, best_i, parts[g].best, parts[g].second, parts[g].best_i);
    assoc_decide(best, second, best_i, *known_count_p, n, j, meas[2 * j], meas[2 * j + 1], state[0], state[1], state[2],
                 state, known_count_p, cmd, assoc_out, dmin_out, second_out, created_out);
}

// local-mode stand-in for the all-reduce of W: dst = sum over shards (rank order)
__global__ void k_sum_shards(double2* __restrict__ dst, const double2* const* __restrict__ srcs, int world, long long ld) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ld) return;
    double2 acc = srcs[0][c];
    for (int g = 1; g < world; ++g) {
        acc.x += srcs[g][c].x;
        acc.y += srcs[g][c].y;
    }
    dst[c] = acc;
}

struct Shard {
    int rank = 0;
    int L0 = 0, L1 = 0;
    long long r0 = 0, r1 = 0;
    int rows = 0;
    double* sig = nullptr;
    double* state = nullptr;
    double2 *K2 = nullptr, *W2 = nullptr, *Wpart = nullptr;
    double* robot = nullptr;  // 3 x ld; aliases sig on the rank that owns rows 0..2
    bool robot_owned = false;
    double *pose0 = nullptr, *motion = nullptr, *meas = nullptr, *xy = nullptr;
    Ctx* ctx = nullptr;
    UpdateCmd* cmd = nullptr;
    AssocPartial *blk = nullptr, *part = nullptr, *parts = nullptr;
    unsigned int* done = nullptr;
    int* known_count = nullptr;
    int32_t* init_flag = nullptr;
    unsigned long long* nupd = nullptr;
    int32_t* d_assoc = nullptr;
    double *d_dmin = nullptr, *d_second = nullptr;
    uint8_t* d_created = nullptr;
    int assoc_blocks = 1;
};

}  // namespace

struct ekf_sharded {
    int n = 0, N = 0, world = 1, device = 0, sm_count = 148;
    bool local = false;
    long long ld = 0;
    std::vector<Shard> sh;  // NCCL mode: exactly this rank's shard; local mode: all of them
    std::vector<long long> r0_of, r1_of;
    ncclComm_t comm = nullptr;
    cudaStream_t stream = nullptr;
    int init_flag_host = 0;
    int pending = 0;  // corrections whose factors are not yet applied to Sigma
    int carry_pending = 1;  // factors may stay pending across prediction() / measurement() calls
    int max_pending = kDefaultPending;  // corrections per sweep (ekf_sharded_set_max_pending)
    uint64_t sweeps = 0;    // passes over Sigma so far
    int m_cap = 0;
    const double2** d_srcs = nullptr;  // local mode: device array of Wpart pointers
    uint64_t launches = 0;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    unsigned char* h_stage = nullptr;  // pinned
    size_t h_stage_bytes = 0;
    // push exchange of W (ekf_sharded_attach_exchange); the buffers belong to the caller
    bool push = false;
    XPeers xp = {};
    unsigned char* xlocal = nullptr;
    unsigned long long gen = 1;     // group generation: what a raised flag holds
    int* d_barrier = nullptr;
    unsigned long long* d_read_count = nullptr;
    unsigned long long corrections_enqueued = 0;
    int rank = 0;
};

namespace {

void partition(ekf_sharded* h) {
    const int per = (h->n + h->world - 1) / h->world;
    h->r0_of.resize(h->world);
    h->r1_of.resize(h->world);
    for (int g = 0; g < h->world; ++g) {
        const int L0 = std::min(h->n, g * per), L1 = std::min(h->n, (g + 1) * per);
        h->r0_of[g] = g == 0 ? 0 : 3 + 2LL * L0;
        h->r1_of[g] = 3 + 2LL * L1;
    }
}

int alloc_shard(ekf_sharded* h, Shard& s, int rank) {
    const int per = (h->n + h->world - 1) / h->world;
    s.rank = rank;
    s.L0 = std::min(h->n, rank * per);
    s.L1 = std::min(h->n, (rank + 1) * per);
    s.r0 = h->r0_of[rank];
    s.r1 = h->r1_of[rank];
    s.rows = (int)(s.r1 - s.r0);
    const size_t ld = (size_t)h->ld;
    CU(cudaMalloc(&s.sig, sizeof(double) * std::max<size_t>(1, (size_t)s.rows) * ld));
    CU(cudaMalloc(&s.state, sizeof(double) * ld));
    CU(cudaMalloc(&s.K2, sizeof(double2) * (ld * kMaxPending + 16)));  // pending factor slots [kMaxPending][ld]
    CU(cudaMalloc(&s.W2, sizeof(double2) * (ld * kMaxPending + 16)));
    CU(cudaMalloc(&s.Wpart, sizeof(double2) * ld));
    if (rank == 0) {
        s.robot = s.sig;
    } else {
        CU(cudaMalloc(&s.robot, sizeof(double) * 3 * ld));
        CU(cudaMemsetAsync(s.robot, 0, sizeof(double) * 3 * ld, h->stream));
        s.robot_owned = true;
    }
    CU(cudaMalloc(&s.pose0, 3 * sizeof(double)));
    CU(cudaMalloc(&s.motion, 2 * sizeof(double)));
    CU(cudaMalloc(&s.xy, sizeof(double) * 2 * h->n));
    CU(cudaMalloc(&s.ctx, sizeof(Ctx)));
    CU(cudaMalloc(&s.cmd, sizeof(UpdateCmd)));
    s.assoc_blocks = std::max(1, std::min((s.L1 - s.L0 + 255) / 256, 1024));
    CU(cudaMalloc(&s.blk, sizeof(AssocPartial) * s.assoc_blocks));
    CU(cudaMalloc(&s.part, sizeof(AssocPartial)));
    CU(cudaMalloc(&s.parts, sizeof(AssocPartial) * h->world));
    CU(cudaMalloc(&s.done, sizeof(unsigned int)));
    CU(cudaMalloc(&s.known_count, sizeof(int)));
    CU(cudaMalloc(&s.init_flag, sizeof(int32_t)));
    CU(cudaMalloc(&s.nupd, sizeof(unsigned long long)));
    CU(cudaMemsetAsync(s.sig, 0, sizeof(double) * std::max<size_t>(1, (size_t)s.rows) * ld, h->stream));
    CU(cudaMemsetAsync(s.state, 0, sizeof(double) * ld, h->stream));
    CU(cudaMemsetAsync(s.K2, 0, sizeof(double2) * ld * kMaxPending, h->stream));
    CU(cudaMemsetAsync(s.W2, 0, sizeof(double2) * ld * kMaxPending, h->stream));
    CU(cudaMemsetAsync(s.Wpart, 0, sizeof(double2) * ld, h->stream));
    CU(cudaMemsetAsync(s.ctx, 0, sizeof(Ctx), h->stream));
    CU(cudaMemsetAsync(s.cmd, 0, sizeof(UpdateCmd), h->stream));
    CU(cudaMemsetAsync(s.done, 0, sizeof(unsigned int), h->stream));
    CU(cudaMemsetAsync(s.known_count, 0, sizeof(int), h->stream));
    CU(cudaMemsetAsync(s.init_flag, 0, sizeof(int32_t), h->stream));
    CU(cudaMemsetAsync(s.nupd, 0, sizeof(unsigned long long), h->stream));
    return 0;  // Sigma0's landmark diagonal (ekf_slam.cpp:29-36) is written by finish_create()
}

__global__ void k_sh_init_sigma(double* __restrict__ sig_local, long long ld, long long r0, int rows) {
    const int lr = blockIdx.x * blockDim.x + threadIdx.x;
    if (lr >= rows) return;
    const long long r = r0 + lr;
    if (r >= 3) sig_local[(long long)lr * ld + r] = kSigma0;
}

int ensure_m(ekf_sharded* h, int m) {
    if (m <= h->m_cap) return 0;
    const int cap = std::max(m, 64);
    CU(cudaStreamSynchronize(h->stream));
    for (auto& s : h->sh) {
        cudaFree(s.meas);
        cudaFree(s.d_assoc);
        cudaFree(s.d_dmin);
        cudaFree(s.d_second);
        cudaFree(s.d_created);
        CU(cudaMalloc(&s.meas, sizeof(double) * 2 * cap));
        CU(cudaMalloc(&s.d_assoc, sizeof(int32_t) * cap));
        CU(cudaMalloc(&s.d_dmin, sizeof(double) * cap));
        CU(cudaMalloc(&s.d_second, sizeof(double) * cap));
        CU(cudaMalloc(&s.d_created, cap));
    }
    const size_t need = (size_t)cap * 64 + (size_t)h->n * 17 + 256;
    if (need > h->h_stage_bytes) {
        if (h->h_stage) cudaFreeHost(h->h_stage);
        h->h_stage = nullptr;
        CU(cudaMallocHost((void**)&h->h_stage, need));
        h->h_stage_bytes = need;
    }
    h->m_cap = cap;
    return 0;
}

// ---- the exchanges
int exchange_W(ekf_sharded* h) {
    if (h->local) {
        const int g = (int)((h->ld + 255) / 256);
        for (auto& s : h->sh) {
            k_sum_shards<<<g, 256, 0, h->stream>>>(s.W2 + (long long)h->pending * h->ld, h->d_srcs, h->world, h->ld);
            h->launches++;
        }
        CU(cudaGetLastError());
    } else {
        Shard& s = h->sh[0];
        NC(ncclAllReduce(s.Wpart, s.W2 + (long long)h->pending * h->ld, 2 * (size_t)h->ld, ncclDouble, ncclSum, h->comm,
                         h->stream));
    }
    return 0;
}
int exchange_robot_rows(ekf_sharded* h) {
    if (h->local) {
        for (size_t g = 1; g < h->sh.size(); ++g)
            CU(cudaMemcpyAsync(h->sh[g].robot, h->sh[0].sig, sizeof(double) * 3 * h->ld, cudaMemcpyDeviceToDevice, h->stream));
    } else {
        Shard& s = h->sh[0];
        NC(ncclBroadcast(s.robot, s.robot, 3 * (size_t)h->ld, ncclDouble, 0, h->comm, h->stream));
    }
    return 0;
}
int exchange_partials(ekf_sharded* h) {
    if (h->local) {
        for (auto& src : h->sh)
            for (auto& dst : h->sh)
                CU(cudaMemcpyAsync(dst.parts + src.rank, src.part, sizeof(AssocPartial), cudaMemcpyDeviceToDevice, h->stream));
    } else {
        Shard& s = h->sh[0];
        NC(ncclAllGather(s.part, s.parts, sizeof(AssocPartial), ncclChar, h->comm, h->stream));
    }
    return 0;
}

// apply the pending factors to every shard's own rows in one sweep
int flush(ekf_sharded* h, int n_counted, bool use_cmd) {
    if (h->pending == 0) return 0;
    if (h->push) {
        // the exchange slots are reused by the next group: no rank may still be reading this group's partials when
        // the first push of the next group lands (a 4-byte all-reduce as the barrier, once per sweep)
        NC(ncclAllReduce(h->d_barrier, h->d_barrier, 1, ncclInt, ncclSum, h->comm, h->stream));
        h->gen += 1;
    }
    for (auto& s : h->sh) {
        if (s.rows > 0) {
            CU(launch_sweep(h->pending, s.sig, h->ld, s.rows, s.K2, s.W2, s.r0, s.nupd, n_counted, use_cmd ? s.cmd : nullptr,
                            h->sm_count, h->stream));
            h->launches++;
        }
    }
    h->pending = 0;
    h->sweeps += 1;
    return 0;
}

// verbs that look at Sigma or at the update counter first bring Sigma up to date
int settle(ekf_sharded* h) { return h->pending ? flush(h, h->pending, false) : 0; }

// one landmark correction across all shards: fills factor slot `pending`; Sigma is swept later (flush)
int correct(ekf_sharded* h, bool use_cmd, bool stale_pose, int lm, double sx, double sy) {
    const int gl = (int)((h->ld + 255) / 256);
    const int p = h->pending;
    if (h->push) {
        Shard& s = h->sh[0];
        h->corrections_enqueued += 1;
        CU(launch_pdl(k_sh_correct_push, dim3(gl), dim3(256), 0, h->stream, (const double*)s.sig, h->ld, s.r0, s.r1, h->r1_of[0], h->N,
                      h->rank, s.state, (const double*)(stale_pose ? s.pose0 : s.state),
                      (const UpdateCmd*)(use_cmd ? s.cmd : nullptr), lm, sx, sy, s.K2, s.W2, p, h->xp,
                      (const unsigned char*)h->xlocal, h->gen, h->d_read_count,
                      h->corrections_enqueued * (unsigned long long)gl));
        h->launches += 1;
        h->pending += 1;
        if (!use_cmd && h->pending >= h->max_pending) return flush(h, h->pending, false);
        return 0;
    }
    for (auto& s : h->sh) {
        k_sh_ctx_h<<<1, 32, 0, h->stream>>>(s.state, stale_pose ? s.pose0 : s.state, use_cmd ? s.cmd : nullptr, lm, sx, sy, s.ctx);
        k_sh_wpart<<<gl, 256, 0, h->stream>>>(s.sig, h->ld, s.r0, s.r1, h->N, s.ctx, s.K2, s.W2, p, s.Wpart);
        h->launches += 2;
    }
    CU(cudaGetLastError());
    int rc = exchange_W(h);
    if (rc) return rc;
    for (auto& s : h->sh) {
        k_sh_gain_state<<<gl, 256, 0, h->stream>>>(s.W2 + (long long)p * h->ld, s.K2 + (long long)p * h->ld, s.state, s.ctx,
                                                   h->N, h->ld);
        h->launches += 1;
    }
    CU(cudaGetLastError());
    h->pending += 1;
    // a correction data_association() may still drop (use_cmd) is flushed by the caller with the command block
    if (!use_cmd && h->pending >= h->max_pending) return flush(h, h->pending, false);
    return 0;
}

int finish_create(ekf_sharded* h) {
    for (auto& s : h->sh)
        if (s.rows > 0) {
            k_sh_init_sigma<<<(s.rows + 255) / 256, 256, 0, h->stream>>>(s.sig, h->ld, s.r0, s.rows);
            h->launches++;
        }
    CU(cudaGetLastError());
    if (h->local) {
        std::vector<const double2*> ptrs;
        for (auto& s : h->sh) ptrs.push_back(s.Wpart);
        CU(cudaMalloc((void**)&h->d_srcs, sizeof(double2*) * ptrs.size()));
        CU(cudaMemcpyAsync((void*)h->d_srcs, ptrs.data(), sizeof(double2*) * ptrs.size(), cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    int rc = ensure_m(h, 64);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

int create_common(int n, int world, int device, ekf_sharded** out, ekf_sharded** hp) {
    if (!out) return fail(-1, "null out pointer");
    *out = nullptr;
    if (n <= 0 || world <= 0 || n < world) return fail(-1, "invalid shape: n=%d world=%d", n, world);
    const int rc = check_device(device);
    if (rc) return rc;
    ekf_sharded* h = new (std::nothrow) ekf_sharded();
    if (!h) return fail(-3, "out of host memory");
    h->n = n;
    h->N = 3 + 2 * n;
    h->world = world;
    h->device = device;
    h->ld = (h->N + 15) & ~15LL;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    partition(h);
    *hp = h;
    return 0;
}

}  // namespace

extern "C" {

const char* ekf_sharded_last_error(void) { return g_err; }

int ekf_sharded_unique_id(void* id128) {
    if (!id128) return fail(-1, "null argument");
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    ncclUniqueId id;
    NC(ncclGetUniqueId(&id));
    memcpy(id128, &id, sizeof(id));
    return 0;
}

int ekf_sharded_destroy(ekf_sharded* h) {
    if (!h) return 0;
    DeviceGuard g(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto& s : h->sh) {
        cudaFree(s.sig);
        cudaFree(s.state);
        cudaFree(s.K2);
        cudaFree(s.W2);
        cudaFree(s.Wpart);
        if (s.robot_owned) cudaFree(s.robot);
        cudaFree(s.pose0);
        cudaFree(s.motion);
        cudaFree(s.meas);
        cudaFree(s.xy);
        cudaFree(s.ctx);
        cudaFree(s.cmd);
        cudaFree(s.blk);
        cudaFree(s.part);
        cudaFree(s.parts);
        cudaFree(s.done);
        cudaFree(s.known_count);
        cudaFree(s.init_flag);
        cudaFree(s.nupd);
        cudaFree(s.d_assoc);
        cudaFree(s.d_dmin);
        cudaFree(s.d_second);
        cudaFree(s.d_created);
    }
    if (h->d_srcs) cudaFree((void*)h->d_srcs);
    cudaFree(h->d_read_count);
    cudaFree(h->d_barrier);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->comm) ncclCommDestroy(h->comm);
    if (h->t0) cudaEventDestroy(h->t0);
    if (h->t1) cudaEventDestroy(h->t1);
    if (h->stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();
    delete h;
    return 0;
}

int ekf_sharded_create(int n, int rank, int world, const void* id128, int device, ekf_sharded** out) {
    if (!id128 || rank < 0 || rank >= world) return fail(-1, "invalid rank / id");
    ekf_sharded* h = nullptr;
    int rc = create_common(n, world, device, out, &h);
    if (rc) return rc;
    DeviceGuard g(device);
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        ekf_sharded_destroy(h);
        return fail((int)e, "stream: %s", cudaGetErrorString(e));
    }
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclResult_t r = ncclCommInitRank(&h->comm, world, id, rank);
    if (r != ncclSuccess) {
        h->comm = nullptr;
        ekf_sharded_destroy(h);
        return fail(1000 + (int)r, "ncclCommInitRank: %s", ncclGetErrorString(r));
    }
    h->rank = rank;
    h->sh.resize(1);
    rc = alloc_shard(h, h->sh[0], rank);
    if (!rc) rc = finish_create(h);
    if (rc) {
        ekf_sharded_destroy(h);
        return rc;
    }
    *out = h;
    return 0;
}

// Push exchange of W (see k_sh_correct_push): the caller provides one symmetric buffer per rank - e.g. from
// torch.distributed._symmetric_memory or cudaIpc handles - of ekf_sharded_exchange_bytes() bytes, zero-filled, mapped
// into this process for every rank (peer_bases[rank'], rank' = 0..world-1), plus the multicast address of the same
// buffer when the fabric has one (0 otherwise).  Collective: every rank attaches before the next verb.  The buffers
// stay the caller's; they must outlive the handle.  Without this call the exchange is an ncclAllReduce.  The call
// fails, and attaches nothing, when the correction kernel's grid cannot be resident at once (ld / 256 CTAs).
#if EKF_SH_PROF
int ekf_sharded_debug_prof(uint64_t* out16) {
    return cudaMemcpyFromSymbol(out16, g_sh_prof, sizeof(uint64_t) * 16) == cudaSuccess ? 0 : -1;
}
#endif
int ekf_sharded_exchange_bytes(ekf_sharded* h, uint64_t* bytes) {
    if (!h || !bytes) return fail(-1, "null argument");
    *bytes = xflag_bytes(h->ld) + (uint64_t)kMaxPending * 2 * (uint64_t)h->ld * sizeof(double2);
    return 0;
}
int ekf_sharded_attach_exchange(ekf_sharded* h, int world, const uint64_t* peer_bases, uint64_t multicast_base) {
    if (!h || !peer_bases) return fail(-1, "null argument");
    if (h->local) return fail(-1, "the push exchange needs real ranks (not the single-GPU emulation)");
    if (world != h->world || world > 8) return fail(-1, "push exchange: world size %d not supported", world);
    DeviceGuard g(h->device);
    {   // k_sh_correct_push's CTAs wait for one another: the whole grid has to be resident at once
        int per_sm = 0;
        CU(kernel_setup<k_sh_correct_push>(h->device, 256, 0, false, &per_sm));
        const long long blocks = (h->ld + 255) / 256;
        if (blocks > (long long)per_sm * h->sm_count)
            return fail(-1, "push exchange: the correction needs %lld resident CTAs, the device holds %d (%d SMs x %d)",
                        blocks, per_sm * h->sm_count, h->sm_count, per_sm);
    }
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    CU(cudaStreamSynchronize(h->stream));
    h->xp = XPeers{};
    for (int r = 0; r < world; ++r) h->xp.base[r] = reinterpret_cast<unsigned char*>((uintptr_t)peer_bases[r]);
    h->xp.mc = reinterpret_cast<unsigned char*>((uintptr_t)multicast_base);
    h->xp.world = world;
    h->xlocal = h->xp.base[h->rank];
    if (!h->d_barrier) {
        CU(cudaMalloc(&h->d_barrier, sizeof(int)));
        CU(cudaMemset(h->d_barrier, 0, sizeof(int)));
        CU(cudaMalloc(&h->d_read_count, sizeof(unsigned long long)));
        CU(cudaMemset(h->d_read_count, 0, sizeof(unsigned long long)));
        h->corrections_enqueued = 0;
    }
    h->gen = 1;
    h->push = true;
    return 0;
}

int ekf_sharded_create_local(int n, int world, int device, ekf_sharded** out) {
    ekf_sharded* h = nullptr;
    int rc = create_common(n, world, device, out, &h);
    if (rc) return rc;
    DeviceGuard g(device);
    h->local = true;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        ekf_sharded_destroy(h);
        return fail((int)e, "stream: %s", cudaGetErrorString(e));
    }
    h->sh.resize(world);
    for (int r = 0; r < world && !rc; ++r) rc = alloc_shard(h, h->sh[r], r);
    if (!rc) rc = finish_create(h);
    if (rc) {
        ekf_sharded_destroy(h);
        return rc;
    }
    *out = h;
    return 0;
}

int ekf_sharded_predict(ekf_sharded* h, double dtheta, double dx) {
    if (!h) return fail(-1, "null handle");
    DeviceGuard g(h->device);
    if (!h->carry_pending) {
        int rc = settle(h);
        if (rc) return rc;
    }
    for (auto& s : h->sh) {
        // on ranks > 0 this updates the copy of rows 0..2, which exchange_robot_rows overwrites before it is read
        k_large_motion<false><<<1, 32, 0, h->stream>>>(s.state, s.robot, h->ld, dtheta, dx, s.motion, s.K2, s.W2,
                                                       h->pending, ref_noise());
        h->launches++;
        int lr_begin = 0;
        if (s.rank == 0) {
            k_sh_predict_rows12<<<(h->N - 3 + 255) / 256, 256, 0, h->stream>>>(s.sig, h->ld, h->N, s.motion);
            h->launches++;
            lr_begin = 3;
        }
        if (s.rows > lr_begin) {
            k_sh_predict_cols<<<(s.rows - lr_begin + 255) / 256, 256, 0, h->stream>>>(s.sig, h->ld, lr_begin, s.rows, s.motion);
            h->launches++;
        }
    }
    CU(cudaGetLastError());
    return 0;
}

int ekf_sharded_measurement(ekf_sharded* h, const double* xy, const uint8_t* visible) {
    if (!h || !xy || !visible) return fail(-1, "null argument");
    DeviceGuard g(h->device);
    const int n = h->n;
    if (!h->init_flag_host) {
        CU(cudaStreamSynchronize(h->stream));
        memcpy(h->h_stage, xy, sizeof(double) * 2 * n);
        for (auto& s : h->sh) {
            CU(cudaMemcpyAsync(s.xy, h->h_stage, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, h->stream));
            k_large_init_landmarks<<<(n + 255) / 256, 256, 0, h->stream>>>(s.state, s.xy, n, s.init_flag);
            h->launches++;
        }
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(h->stream));
        h->init_flag_host = 1;
    }
    for (auto& s : h->sh) CU(cudaMemcpyAsync(s.pose0, s.state, 3 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    for (int i = 0; i < n; ++i) {
        if (!visible[i]) continue;
        int rc = correct(h, false, true, i, xy[2 * i], xy[2 * i + 1]);
        if (rc) return rc;
    }
    return h->carry_pending ? 0 : flush(h, h->pending, false);
}

int ekf_sharded_data_association(ekf_sharded* h, const double* xy, int m, uint8_t* known, int32_t* assoc_out,
                                 double* dmin_out, double* second_out, uint8_t* created_out) {
    if (!h || !known || m < 0 || (m > 0 && !xy)) return fail(-1, "invalid argument");
    if (m == 0) return 0;
    DeviceGuard g(h->device);
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    const int n = h->n;
    int rc = ensure_m(h, m);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    int known_count = 0;
    while (known_count < n && known[known_count]) ++known_count;
    double* st_xy = reinterpret_cast<double*>(h->h_stage);
    memcpy(st_xy, xy, sizeof(double) * 2 * m);
    int* st_kc = reinterpret_cast<int*>(h->h_stage + sizeof(double) * 2 * m);
    *st_kc = known_count;
    for (auto& s : h->sh) {
        CU(cudaMemcpyAsync(s.meas, st_xy, sizeof(double) * 2 * m, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(s.known_count, st_kc, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    }
    for (int j = 0; j < m; ++j) {
        rc = exchange_robot_rows(h);
        if (rc) return rc;
        for (auto& s : h->sh) {
            k_sh_assoc_local<<<s.assoc_blocks, 256, 0, h->stream>>>(s.robot, s.sig, h->ld, s.r0, s.L0, s.L1, s.state, s.meas, j,
                                                                     s.known_count, s.blk, s.done, s.part);
            h->launches++;
        }
        CU(cudaGetLastError());
        rc = exchange_partials(h);
        if (rc) return rc;
        for (auto& s : h->sh) {
            k_sh_decide<<<1, 32, 0, h->stream>>>(s.parts, h->world, s.state, n, s.meas, j, s.known_count, s.cmd, s.d_assoc,
                                                 s.d_dmin, s.d_second, s.d_created);
            h->launches++;
        }
        CU(cudaGetLastError());
        rc = correct(h, true, false, 0, 0.0, 0.0);
        if (rc) return rc;
        rc = flush(h, 1, true);  // the next measurement's distances need the corrected Sigma
        if (rc) return rc;
    }
    Shard& s0 = h->sh[0];  // every replica holds the same decisions
    unsigned char* o = h->h_stage + sizeof(double) * 2 * m + 64;
    int32_t* o_assoc = reinterpret_cast<int32_t*>(o);
    double* o_dmin = reinterpret_cast<double*>(o + (((size_t)m * 4 + 15) & ~(size_t)15));
    double* o_second = o_dmin + m;
    uint8_t* o_created = reinterpret_cast<uint8_t*>(o_second + m);
    int* o_kc = reinterpret_cast<int*>(o_created + ((m + 15) & ~15));
    CU(cudaMemcpyAsync(o_assoc, s0.d_assoc, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(o_dmin, s0.d_dmin, sizeof(double) * m, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(o_second, s0.d_second, sizeof(double) * m, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(o_created, s0.d_created, m, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(o_kc, s0.known_count, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (assoc_out) memcpy(assoc_out, o_assoc, sizeof(int32_t) * m);
    if (dmin_out) memcpy(dmin_out, o_dmin, sizeof(double) * m);
    if (second_out) memcpy(second_out, o_second, sizeof(double) * m);
    if (created_out) memcpy(created_out, o_created, m);
    for (int i = known_count; i < *o_kc && i < n; ++i) known[i] = 1;
    return 0;
}

int ekf_sharded_get_state(ekf_sharded* h, double* out) {
    if (!h || !out) return fail(-1, "null argument");
    DeviceGuard g(h->device);
    CU(cudaMemcpyAsync(out, h->sh[0].state, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}
int ekf_sharded_rows(ekf_sharded* h, int shard, int64_t* row_begin, int64_t* row_end) {
    if (!h || shard < 0 || shard >= (int)h->sh.size()) return fail(-1, "invalid shard");
    if (row_begin) *row_begin = h->sh[shard].r0;
    if (row_end) *row_end = h->sh[shard].r1;
    return 0;
}
int ekf_sharded_get_sigma_rows(ekf_sharded* h, int shard, double* out, int64_t ld) {
    if (!h || !out || shard < 0 || shard >= (int)h->sh.size() || ld < h->N) return fail(-1, "invalid argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    Shard& s = h->sh[shard];
    if (s.rows > 0)
        CU(cudaMemcpy2DAsync(out, sizeof(double) * ld, s.sig, sizeof(double) * h->ld, sizeof(double) * h->N, s.rows,
                             cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}
// Selected GLOBAL rows owned by shard `shard` (NCCL mode: 0 = this rank), N doubles each, row stride ld in `out`.
int ekf_sharded_get_sigma_row_list(ekf_sharded* h, int shard, const int64_t* rows, int count, double* out, int64_t ld) {
    if (!h || shard < 0 || shard >= (int)h->sh.size() || count < 0 || (count > 0 && (!rows || !out)) || ld < h->N)
        return fail(-1, "invalid argument");
    Shard& s = h->sh[shard];
    for (int k = 0; k < count; ++k)
        if (rows[k] < s.r0 || rows[k] >= s.r1) return fail(-1, "row %lld is not owned by this shard", (long long)rows[k]);
    DeviceGuard g(h->device);
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    for (int k = 0; k < count; ++k)
        CU(cudaMemcpyAsync(out + (size_t)k * ld, s.sig + (size_t)(rows[k] - s.r0) * h->ld, sizeof(double) * h->N,
                           cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}
int ekf_sharded_update_count(ekf_sharded* h, uint64_t* out) {
    if (!h || !out) return fail(-1, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, h->sh[0].nupd, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    *out = v;
    return 0;
}
int ekf_sharded_set_max_pending(ekf_sharded* h, int max_pending) {
    if (!h || max_pending < 1 || max_pending > kMaxPending) return fail(-1, "max_pending must be 1..%d", kMaxPending);
    DeviceGuard g(h->device);
    h->max_pending = max_pending;
    return h->pending >= max_pending ? settle(h) : 0;
}
int ekf_sharded_sweep_count(ekf_sharded* h, uint64_t* out) {
    if (!h || !out) return fail(-1, "null argument");
    *out = h->sweeps;
    return 0;
}
int ekf_sharded_set_carry_pending(ekf_sharded* h, int carry) {
    if (!h) return fail(-1, "null handle");
    h->carry_pending = carry ? 1 : 0;
    if (!h->carry_pending) {
        DeviceGuard g(h->device);
        return settle(h);
    }
    return 0;
}
int ekf_sharded_launch_count(ekf_sharded* h, uint64_t* out) {
    if (!h || !out) return fail(-1, "null argument");
    *out = h->launches;
    return 0;
}
int ekf_sharded_sync(ekf_sharded* h) {
    if (!h) return fail(-1, "null handle");
    DeviceGuard g(h->device);
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}
int ekf_sharded_timer_start(ekf_sharded* h) {
    if (!h) return fail(-1, "null handle");
    DeviceGuard g(h->device);
    if (!h->t0) {
        CU(cudaEventCreate(&h->t0));
        CU(cudaEventCreate(&h->t1));
    }
    CU(cudaEventRecord(h->t0, h->stream));
    return 0;
}
int ekf_sharded_timer_stop(ekf_sharded* h, float* ms_out) {
    if (!h || !ms_out || !h->t0) return fail(-1, "timer not started");
    DeviceGuard g(h->device);
    {
        int rc_ = settle(h);
        if (rc_) return rc_;
    }
    CU(cudaEventRecord(h->t1, h->stream));
    CU(cudaEventSynchronize(h->t1));
    CU(cudaEventElapsedTime(ms_out, h->t0, h->t1));
    return 0;
}

}  // extern "C"
