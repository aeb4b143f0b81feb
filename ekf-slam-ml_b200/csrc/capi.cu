// Host side of the C ABI declared in include/ekf_slam_b200.h: handle management, staging, kernel
// launches.  No algorithmic work happens on the host — there is deliberately no CPU fallback.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <new>
#include <vector>

#include "../../include/ekf_slam_b200.h"
#include "ekf_fused.cuh"
#include "ekf_fused_sym.cuh"
#include "ekf_fused_tile.cuh"
#include "ekf_batch_wide.cuh"
#include "ekf_batch_consistency.cuh"
#include "ekf_large.cuh"
#include "ekf_large_mma.cuh"
#include "host_util.cuh"

using namespace ekf;

namespace {

constexpr int kFusedMaxN = 64;  // landmarks; Sigma (131^2 fp64 = 137 KB) must fit shared memory
constexpr int kRing = 8;

int max_smem_optin(int device) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    return v;
}

// Launch one of the shared-memory kernels (ekf_fused_kernel, ekf_fused_sym_kernel): one single-warp CTA per filter
// with `smem` bytes of shared memory.
template <void (*Kernel)(FusedParams)>
int launch_smem_kernel(int smem, const FusedParams& p, cudaStream_t stream, int device) {
    if (smem > max_smem_optin(device))
        return fail(EKF_ERR_UNSUPPORTED, "fused engine: %d B of shared memory needed for n=%d", smem, p.n);
    if (p.B <= 0) return EKF_OK;
    CU(kernel_setup<Kernel>(device, 32, smem, true));
    Kernel<<<(unsigned)p.B, 32, smem, stream>>>(p);
    CU(cudaGetLastError());
    return EKF_OK;
}

// Single filter: dense Sigma (ekf_fused.cuh); n = 20 gets the fully unrolled rank-2 pass.
int launch_fused(const FusedParams& p, cudaStream_t stream, int device) {
    const int smem = FusedSmem(p.n, p.m_max).total;
    return p.n == 20 ? launch_smem_kernel<ekf_fused_kernel<20>>(smem, p, stream, device)
                     : launch_smem_kernel<ekf_fused_kernel<0>>(smem, p, stream, device);
}

// Batch with n <= 64, n != 20: symmetric staircase Sigma (ekf_fused_sym.cuh).
int launch_fused_staircase(const FusedParams& p, cudaStream_t stream, int device) {
    const int smem = SymSmem(p.n, p.m_max, p.nis != nullptr).total;
    return p.nis ? launch_smem_kernel<ekf_fused_sym_kernel<true>>(smem, p, stream, device)
                 : launch_smem_kernel<ekf_fused_sym_kernel<false>>(smem, p, stream, device);
}

// Batched engine at the reference's map size (n = 20): Sigma resident in registers (ekf_fused_tile.cuh).
template <bool Assoc, bool Nis>
int launch_fused_tile(const FusedParams& p, cudaStream_t stream, int device, int sm_count) {
    const tile::TileSmem L(p.m_max, Assoc, Nis);
    if (L.total > max_smem_optin(device))
        return fail(EKF_ERR_UNSUPPORTED, "fused engine: %d B of shared memory needed for m_max=%d", L.total, p.m_max);
    if (p.sig_stride != tile::kStride || p.st_stride != tile::kStride || p.n != tile::kNL ||
        p.state != p.sigma + tile::kStOff)
        return fail(EKF_ERR_STATE, "tile engine: unexpected batch layout");
    if (p.B <= 0) return EKF_OK;
    // persistent warps: as many single-warp CTAs as fit the device at once, each walking filters b, b + grid, ...
    int per_sm = 0;
    CU((kernel_setup<tile::ekf_fused_tile_kernel<Assoc, Nis>>(device, 32, L.total, true, &per_sm)));
    const long long resident = (long long)sm_count * std::max(per_sm, 1);
    tile::ekf_fused_tile_kernel<Assoc, Nis><<<(unsigned)std::min<long long>(p.B, resident), 32, L.total, stream>>>(p);
    CU(cudaGetLastError());
    return EKF_OK;
}

// Sigma0 = blockdiag(0_3, 100 I) (ekf_slam.cpp:29-36) for B filters of an already-zeroed buffer: dense rows of stride
// ld, one filter every `stride` doubles.
__global__ void k_init_sigma(double* __restrict__ sigma, long long B, int N, long long ld, long long stride) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * (N - 3)) return;
    const long long b = e / (N - 3), k = 3 + e - b * (N - 3);
    sigma[b * stride + k * ld + k] = kSigma0;
}

__global__ void k_maha_one(const double* sig, long long ld, const double* state, int i, double sx, double sy,
                           double* out) {
    double zr, zphi;
    range_bearing(sx, sy, zr, zphi);
    *out = maha_distance(sig, ld, i, state[3 + 2 * i], state[4 + 2 * i], zr, zphi, state[0], state[1], state[2]);
}

__global__ void k_update_pose(double wheel_base, double wheel_radius, long long count, double* poses,
                              const double* left, const double* right) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    double x = poses[3 * k], y = poses[3 * k + 1], th = poses[3 * k + 2];
    update_pose(wheel_base, wheel_radius, left[k], right[k], x, y, th);
    poses[3 * k] = x, poses[3 * k + 1] = y, poses[3 * k + 2] = th;
}

__global__ void k_normalize(const double* in, double* out, long long count) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < count) out[k] = normalize_angle(in[k]);
}

__global__ void k_gather_poses(const double* state, long long B, int st_stride, double* out) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= 3 * B) return;
    const long long b = k / 3;
    out[k] = state[b * st_stride + (k - 3 * b)];
}

// truth[b] = {x, y, theta}; state = {theta, x, y}
__global__ void k_pose_error(const double* state, long long B, int st_stride, const double* truth, double* acc4) {
    double ex = 0, ey = 0, et = 0;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const double* s = state + b * st_stride;
        const double dx = s[1] - truth[3 * b], dy = s[2] - truth[3 * b + 1];
        const double dt = normalize_angle(s[0] - truth[3 * b + 2]);
        ex += dx * dx;
        ey += dy * dy;
        et += dt * dt;
    }
    for (int off = 16; off > 0; off >>= 1) {
        ex += __shfl_xor_sync(0xffffffffu, ex, off);
        ey += __shfl_xor_sync(0xffffffffu, ey, off);
        et += __shfl_xor_sync(0xffffffffu, et, off);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(acc4 + 0, ex);
        atomicAdd(acc4 + 1, ey);
        atomicAdd(acc4 + 2, et);
    }
}

}  // namespace

// ======================================================================================= handles
struct ekf_filter {
    FILE* assoc_log = nullptr;     // ekf_association_log_open(): one line per associated measurement
    uint64_t assoc_calls = 0;      // data_association() calls so far (the log's first column)
    int n = 0, N = 0, device = 0, engine = 0;
    cudaStream_t stream = nullptr;
    uint64_t launches = 0;
    // persistent filter state
    double* d_sigma = nullptr;
    long long ld = 0;          // row stride (stream engine: padded; fused engine: N)
    long long sig_elems = 0;   // allocated doubles
    double* d_state = nullptr;
    int st_stride = 0;
    int32_t* d_init_flag = nullptr;
    unsigned long long* d_nupd = nullptr;
    int init_flag_host = 0;  // mirror used by the stream engine's host-side sequencing
    // inputs / outputs on the device
    int m_cap = 0;
    double* d_in = nullptr;       // xy (2n) or meas (2 m_cap)
    uint8_t* d_flags = nullptr;   // visible (n) / known (n)
    int32_t* d_assoc = nullptr;
    double* d_dmin = nullptr;
    double* d_second = nullptr;
    uint8_t* d_created = nullptr;
    double* d_scalar = nullptr;  // maha out
    // pinned staging ring
    unsigned char* h_ring[kRing] = {nullptr};
    cudaEvent_t ring_ev[kRing] = {nullptr};
    size_t ring_bytes = 0;
    int ring_pos = 0;
    unsigned char* h_out = nullptr;  // pinned output staging
    // Fused engine: the kernels read their inputs from the pinned ring and leave the pose in h_pose through the
    // device mapping of that memory (no copy commands on the stream; a step is launch + synchronise).
    double* h_pose = nullptr;
    // prediction() on the small engine is deferred: the twist waits here and rides along with the next measurement() /
    // data_association() kernel (mode kDoPredict | ...), one launch and one round trip of Sigma instead of two; any other
    // verb that looks at or changes the filter applies it first (stream_settle).
    bool pred_pending = false;
    double pred_tw[2] = {0.0, 0.0};
    bool pose_host_ok = false;  // h_pose holds the pose of the last enqueued kernel
    bool external = false;      // ekf_device_pointers() handed the state out: h_pose can no longer be trusted
    size_t h_out_bytes = 0;
    // stream engine scratch
    double2* d_K2 = nullptr;  // [kMaxPending][ld] pending gain factors
    double2* d_W2 = nullptr;  // [kMaxPending][ld] pending H*Sigma factors
    double* d_state_alt = nullptr;  // ping-pong partner of d_state (the gain kernel never writes what it reads)
    int pending = 0;                // corrections computed but not yet applied to Sigma
    int max_pending = kDefaultPending;  // flush threshold (1 = the reference's one sweep per correction)
    int carry_pending = 1;          // factors may stay pending across prediction() / measurement() calls
    uint64_t sweeps = 0;            // passes over Sigma so far (streamed engine)
    double* d_motion = nullptr;
    double* d_pose0 = nullptr;
    UpdateCmd* d_cmd = nullptr;
    AssocPartial* d_partials = nullptr;
    unsigned int* d_done = nullptr;
    int* d_known_count = nullptr;
    int assoc_blocks = 0;
    int sm_count = 148;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
};

namespace {

int free_filter(ekf_filter* h) {
    if (!h) return EKF_OK;
    if (h->assoc_log) fclose(h->assoc_log);
    h->assoc_log = nullptr;
    DeviceGuard g(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_sigma);
    cudaFree(h->d_state);
    cudaFree(h->d_init_flag);
    cudaFree(h->d_nupd);
    cudaFree(h->d_in);
    cudaFree(h->d_flags);
    cudaFree(h->d_assoc);
    cudaFree(h->d_dmin);
    cudaFree(h->d_second);
    cudaFree(h->d_created);
    cudaFree(h->d_scalar);
    cudaFree(h->d_K2);
    cudaFree(h->d_W2);
    cudaFree(h->d_state_alt);
    cudaFree(h->d_motion);
    cudaFree(h->d_pose0);
    cudaFree(h->d_cmd);
    cudaFree(h->d_partials);
    cudaFree(h->d_done);
    cudaFree(h->d_known_count);
    for (int i = 0; i < kRing; ++i) {
        if (h->h_ring[i]) cudaFreeHost(h->h_ring[i]);
        if (h->ring_ev[i]) cudaEventDestroy(h->ring_ev[i]);
    }
    if (h->h_out) cudaFreeHost(h->h_out);
    if (h->h_pose) cudaFreeHost(h->h_pose);
    if (h->t0) cudaEventDestroy(h->t0);
    if (h->t1) cudaEventDestroy(h->t1);
    if (h->stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();
    delete h;
    return EKF_OK;
}

// (re)size the measurement-count dependent buffers
int ensure_m_cap(ekf_filter* h, int m) {
    if (m <= h->m_cap) return EKF_OK;
    const int cap = std::max(std::max(m, h->n), 32);
    cudaStreamSynchronize(h->stream);
    cudaFree(h->d_in);
    cudaFree(h->d_assoc);
    cudaFree(h->d_dmin);
    cudaFree(h->d_second);
    cudaFree(h->d_created);
    h->d_in = nullptr;
    h->d_assoc = nullptr;
    h->d_dmin = h->d_second = nullptr;
    h->d_created = nullptr;
    CU(cudaMalloc(&h->d_in, sizeof(double) * 2 * cap));
    CU(cudaMalloc(&h->d_assoc, sizeof(int32_t) * cap));
    CU(cudaMalloc(&h->d_dmin, sizeof(double) * cap));
    CU(cudaMalloc(&h->d_second, sizeof(double) * cap));
    CU(cudaMalloc(&h->d_created, cap));
    const size_t need = sizeof(double) * 2 * cap + h->n + 64;
    if (need > h->ring_bytes) {
        for (int i = 0; i < kRing; ++i) {
            if (h->h_ring[i]) cudaFreeHost(h->h_ring[i]);
            h->h_ring[i] = nullptr;
            CU(cudaMallocHost((void**)&h->h_ring[i], need));
        }
        h->ring_bytes = need;
    }
    const size_t out_need = (size_t)cap * (sizeof(int32_t) + 2 * sizeof(double) + 1) + (size_t)h->n + 64 +
                            sizeof(double) * (size_t)h->N;
    if (out_need > h->h_out_bytes) {
        if (h->h_out) cudaFreeHost(h->h_out);
        h->h_out = nullptr;
        CU(cudaMallocHost((void**)&h->h_out, out_need));
        h->h_out_bytes = out_need;
    }
    h->m_cap = cap;
    return EKF_OK;
}

// next pinned staging slot, safe to overwrite
int ring_acquire(ekf_filter* h, unsigned char** slot, cudaEvent_t* ev) {
    const int i = h->ring_pos;
    h->ring_pos = (i + 1) % kRing;
    CU(cudaEventSynchronize(h->ring_ev[i]));
    *slot = h->h_ring[i];
    *ev = h->ring_ev[i];
    return EKF_OK;
}

// The filter's own buffers; each verb points the inputs and outputs of its mode at its pinned slot.
FusedParams fused_params(ekf_filter* h, int mode, int m_max) {
    FusedParams p;
    memset(&p, 0, sizeof(p));
    p.sigma = h->d_sigma;
    p.state = h->d_state;
    p.init_flag = h->d_init_flag;
    p.n_updates = h->d_nupd;
    p.pose_out = h->h_pose;
    p.B = 1;
    p.n = h->n;
    p.m_max = m_max;
    p.mode = mode;
    p.sig_stride = (int)h->sig_elems;
    p.st_stride = h->st_stride;
    return p;
}

// Apply the pending factors to Sigma in one sweep (ekf_large_delayed.cuh).
int stream_flush(ekf_filter* h, int n_counted, const UpdateCmd* cmd) {
    if (h->pending == 0) return EKF_OK;
    CU(launch_sweep(h->pending, h->d_sigma, h->ld, h->N, h->d_K2, h->d_W2, 0, h->d_nupd, n_counted, cmd, h->sm_count,
                    h->stream));
    h->launches += 1;
    h->sweeps += 1;
    h->pending = 0;
    return EKF_OK;
}

// One landmark correction on the stream engine: the gain kernel appends a factor pair; Sigma itself is only
// touched when kMaxPending factors have piled up or the verb ends.
int stream_correct(ekf_filter* h, const double* pose_src, const UpdateCmd* cmd, int lm, double sx, double sy) {
    const int gb = (int)((h->ld + 255) / 256);
    CU(launch_pdl(k_large_gain_p, dim3(gb), dim3(kGainThreads), 0, h->stream, h->d_sigma, h->ld, h->N, h->d_state, h->d_state_alt,
                  pose_src, cmd, lm, sx, sy, h->d_K2, h->d_W2, h->pending));
    h->launches += 1;
    std::swap(h->d_state, h->d_state_alt);
    h->pending += 1;
    // a correction that data_association() may still drop (cmd != nullptr) is flushed by the caller, which passes
    // the command block so that the sweep is skipped and the update not counted for a dropped measurement
    if (!cmd && h->pending >= h->max_pending) return stream_flush(h, h->pending, nullptr);
    return EKF_OK;
}

// Verbs that look at Sigma or at the update counter first bring Sigma up to date (factors may stay pending across
// prediction() and measurement() calls).
int fused_flush_predict(ekf_filter* h) {
    if (!h->pred_pending) return EKF_OK;
    unsigned char* slot;
    cudaEvent_t ev;
    int rc = ring_acquire(h, &slot, &ev);
    if (rc) return rc;
    double* tw = reinterpret_cast<double*>(slot);
    tw[0] = h->pred_tw[0];
    tw[1] = h->pred_tw[1];
    FusedParams p = fused_params(h, kDoPredict, 1);
    p.twists = tw;  // read through the device mapping of the pinned slot
    rc = launch_fused(p, h->stream, h->device);
    CU(cudaEventRecord(ev, h->stream));
    h->launches += 1;
    h->pose_host_ok = rc == EKF_OK;
    h->pred_pending = false;
    return rc;
}

// verbs that only look at the state vector: the streamed engine's pending Sigma factors may stay pending
int settle_prediction(ekf_filter* h) { return h->engine == EKF_ENGINE_FUSED ? fused_flush_predict(h) : EKF_OK; }

int stream_settle(ekf_filter* h) {
    if (h->engine == EKF_ENGINE_FUSED) return fused_flush_predict(h);
    if (h->pending == 0) return EKF_OK;
    return stream_flush(h, h->pending, nullptr);
}

// Buffers and initial state (Sigma0, zero state) of a new filter; on failure the caller frees the half-made handle.
int alloc_filter(ekf_filter* h) {
    const int n = h->n;
    CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    for (int i = 0; i < kRing; ++i) CU(cudaEventCreateWithFlags(&h->ring_ev[i], cudaEventDisableTiming));
    h->st_stride = fused_round16(h->N);
    if (h->engine == EKF_ENGINE_FUSED) {
        h->ld = h->N;
        h->sig_elems = fused_round16(h->N * h->N);
    } else {
        h->ld = fused_round16(h->N);
        h->sig_elems = (long long)h->N * h->ld;
    }
    CU(cudaMalloc(&h->d_sigma, sizeof(double) * (size_t)h->sig_elems));
    CU(cudaMalloc(&h->d_state, sizeof(double) * h->st_stride));
    CU(cudaMalloc(&h->d_init_flag, sizeof(int32_t)));
    CU(cudaMalloc(&h->d_nupd, sizeof(unsigned long long)));
    CU(cudaMalloc(&h->d_flags, (size_t)n + 16));
    CU(cudaMalloc(&h->d_scalar, sizeof(double)));
    CU(cudaMemsetAsync(h->d_nupd, 0, sizeof(unsigned long long), h->stream));
    CU(cudaMemsetAsync(h->d_sigma, 0, sizeof(double) * (size_t)h->sig_elems, h->stream));
    CU(cudaMemsetAsync(h->d_state, 0, sizeof(double) * h->st_stride, h->stream));
    CU(cudaMemsetAsync(h->d_init_flag, 0, sizeof(int32_t), h->stream));
    k_init_sigma<<<(h->N - 3 + 255) / 256, 256, 0, h->stream>>>(h->d_sigma, 1, h->N, h->ld, h->sig_elems);
    h->launches += 1;
    CU(cudaGetLastError());
    if (h->engine == EKF_ENGINE_FUSED) {
        CU(cudaMallocHost((void**)&h->h_pose, 64));
    } else {
        CU(cudaMalloc(&h->d_K2, sizeof(double2) * ((size_t)h->ld * kMaxPending + 16)));
        CU(cudaMalloc(&h->d_W2, sizeof(double2) * ((size_t)h->ld * kMaxPending + 16)));
        CU(cudaMalloc(&h->d_state_alt, sizeof(double) * h->st_stride));
        CU(cudaMemsetAsync(h->d_state_alt, 0, sizeof(double) * h->st_stride, h->stream));
        CU(cudaMalloc(&h->d_motion, 2 * sizeof(double)));
        CU(cudaMalloc(&h->d_pose0, 3 * sizeof(double)));
        CU(cudaMalloc(&h->d_cmd, sizeof(UpdateCmd)));
        h->assoc_blocks = std::max(1, std::min((n + 255) / 256, 1024));
        CU(cudaMalloc(&h->d_partials, sizeof(AssocPartial) * h->assoc_blocks));
        CU(cudaMalloc(&h->d_done, sizeof(unsigned int)));
        CU(cudaMalloc(&h->d_known_count, sizeof(int)));
        CU(cudaMemsetAsync(h->d_done, 0, sizeof(unsigned int), h->stream));
        CU(cudaMemsetAsync(h->d_cmd, 0, sizeof(UpdateCmd), h->stream));
        CU(cudaMemsetAsync(h->d_K2, 0, sizeof(double2) * (size_t)h->ld * kMaxPending, h->stream));
        CU(cudaMemsetAsync(h->d_W2, 0, sizeof(double2) * (size_t)h->ld * kMaxPending, h->stream));
    }
    int rc = ensure_m_cap(h, std::max(n, 32));
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}

}  // namespace

extern "C" {

const char* ekf_version(void) { return "ekf-slam-ml_b200 0.1 (sm_100a)"; }
const char* ekf_last_error(void) { return g_err; }

int ekf_device_count(int* count_out) {
    if (!count_out) return fail(EKF_ERR_INVALID, "null argument");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *count_out = 0;
        return fail((int)e, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *count_out = c;
    return EKF_OK;
}

int ekf_host_alloc(void** out, uint64_t bytes) {
    if (!out) return fail(EKF_ERR_INVALID, "null argument");
    CU(cudaMallocHost(out, bytes ? bytes : 1));
    return EKF_OK;
}
int ekf_host_free(void* p) {
    if (p) CU(cudaFreeHost(p));
    return EKF_OK;
}

int ekf_create_ex(int n, int device, int engine, ekf_filter** out) {
    if (!out) return fail(EKF_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (n <= 0 || n > 500000) return fail(EKF_ERR_INVALID, "n_landmarks=%d out of range", n);
    int rc = check_device(device);
    if (rc) return rc;
    if (engine == EKF_ENGINE_AUTO) engine = (n <= kFusedMaxN) ? EKF_ENGINE_FUSED : EKF_ENGINE_STREAM;
    if (engine != EKF_ENGINE_FUSED && engine != EKF_ENGINE_STREAM) return fail(EKF_ERR_INVALID, "unknown engine %d", engine);
    if (engine == EKF_ENGINE_FUSED && n > kFusedMaxN)
        return fail(EKF_ERR_UNSUPPORTED, "fused engine supports n <= %d", kFusedMaxN);
    DeviceGuard g(device);
    ekf_filter* h = new (std::nothrow) ekf_filter();
    if (!h) return fail(EKF_ERR_STATE, "out of host memory");
    h->n = n;
    h->N = 3 + 2 * n;
    h->device = device;
    h->engine = engine;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    rc = alloc_filter(h);
    if (rc) {
        free_filter(h);
        return rc;
    }
    *out = h;
    return EKF_OK;
}

int ekf_create(int n, int device, ekf_filter** out) { return ekf_create_ex(n, device, EKF_ENGINE_AUTO, out); }

int ekf_clone(ekf_filter* src, ekf_filter** out) {
    if (!src || !out) return fail(EKF_ERR_INVALID, "null argument");
    int rc = ekf_create_ex(src->n, src->device, src->engine, out);
    if (rc) return rc;
    ekf_filter* h = *out;
    DeviceGuard g(src->device);
    // a half-made copy must not reach the caller: any failure below destroys it and clears *out
    rc = stream_settle(src);
    cudaError_t e = cudaSuccess;
    if (!rc) e = cudaStreamSynchronize(src->stream);
    if (!rc && e == cudaSuccess)
        e = cudaMemcpy(h->d_sigma, src->d_sigma, sizeof(double) * (size_t)src->sig_elems, cudaMemcpyDeviceToDevice);
    if (!rc && e == cudaSuccess)
        e = cudaMemcpy(h->d_state, src->d_state, sizeof(double) * src->st_stride, cudaMemcpyDeviceToDevice);
    if (!rc && e == cudaSuccess)
        e = cudaMemcpy(h->d_init_flag, src->d_init_flag, sizeof(int32_t), cudaMemcpyDeviceToDevice);
    if (!rc && e == cudaSuccess)
        e = cudaMemcpy(h->d_nupd, src->d_nupd, sizeof(unsigned long long), cudaMemcpyDeviceToDevice);
    if (!rc && e != cudaSuccess) {
        cudaGetLastError();
        rc = fail((int)e, "ekf_clone: %s", cudaGetErrorString(e));
    }
    if (rc) {
        free_filter(h);
        *out = nullptr;
        return rc;
    }
    h->init_flag_host = src->init_flag_host;
    h->max_pending = src->max_pending;
    h->carry_pending = src->carry_pending;
    return EKF_OK;
}

int ekf_destroy(ekf_filter* h) { return free_filter(h); }
int ekf_num_landmarks(const ekf_filter* h) { return h ? h->n : EKF_ERR_INVALID; }
int ekf_engine(const ekf_filter* h) { return h ? h->engine : EKF_ERR_INVALID; }
void* ekf_stream(ekf_filter* h) { return h ? (void*)h->stream : nullptr; }

int ekf_predict(ekf_filter* h, double dtheta, double dx) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    if (h->engine == EKF_ENGINE_FUSED) {
        int rc = fused_flush_predict(h);  // two predictions in a row: the earlier one goes first, on its own
        if (rc) return rc;
        h->pred_tw[0] = dtheta;
        h->pred_tw[1] = dx;
        h->pred_pending = true;
        return EKF_OK;
    }
    if (h->pending > 0 && !h->carry_pending) {
        int rc = stream_flush(h, h->pending, nullptr);
        if (rc) return rc;
    }
    // motion model + robot block + the pending factors carried across the prediction (ekf_large_delayed.cuh), then
    // the robot-landmark strips
    CU(launch_pdl(k_large_motion, dim3(1), dim3(32), 0, h->stream, h->d_state, h->d_sigma, h->ld, dtheta, dx, h->d_motion,
                  h->d_K2, h->d_W2, h->pending));
    CU(launch_pdl(k_large_predict_strips, dim3((h->N - 3 + 255) / 256), dim3(256), 0, h->stream, h->d_sigma, h->ld, h->N,
                  (const double*)h->d_motion));
    h->launches += 2;
    return EKF_OK;
}

int ekf_measurement(ekf_filter* h, const double* xy, const uint8_t* visible) {
    if (!h || !xy || !visible) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    const int n = h->n;
    if (h->engine == EKF_ENGINE_FUSED) {
        unsigned char* slot;
        cudaEvent_t ev;
        int rc = ring_acquire(h, &slot, &ev);
        if (rc) return rc;
        memcpy(slot, xy, sizeof(double) * 2 * n);
        memcpy(slot + sizeof(double) * 2 * n, visible, n);
        double* tw = reinterpret_cast<double*>(slot + sizeof(double) * 2 * n + ((n + 7) & ~7));
        tw[0] = h->pred_tw[0];
        tw[1] = h->pred_tw[1];
        FusedParams p = fused_params(h, kDoMeasurement | (h->pred_pending ? kDoPredict : 0), 1);
        h->pred_pending = false;
        p.twists = tw;
        p.xy = reinterpret_cast<const double*>(slot);
        p.vis = slot + sizeof(double) * 2 * n;
        rc = launch_fused(p, h->stream, h->device);
        CU(cudaEventRecord(ev, h->stream));
        h->launches += 1;
        h->pose_host_ok = rc == EKF_OK;
        return rc;
    }
    // stream engine: the host sequences one (gain, sweep) pair per visible landmark; readings travel as kernel
    // arguments, the entry-time pose is snapshotted on the device (ekf_slam.cpp:109-111).
    if (!h->init_flag_host) {
        unsigned char* slot;
        cudaEvent_t ev;
        int rc = ring_acquire(h, &slot, &ev);
        if (rc) return rc;
        memcpy(slot, xy, sizeof(double) * 2 * n);
        CU(cudaMemcpyAsync(h->d_in, slot, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, h->stream));
        CU(cudaEventRecord(ev, h->stream));
        k_large_init_landmarks<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_state, h->d_in, n, h->d_init_flag);
        h->launches += 1;
        h->init_flag_host = 1;
    }
    CU(cudaMemcpyAsync(h->d_pose0, h->d_state, 3 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    for (int i = 0; i < n; ++i) {
        if (!visible[i]) continue;
        int rc = stream_correct(h, h->d_pose0, nullptr, i, xy[2 * i], xy[2 * i + 1]);
        if (rc) return rc;
    }
    // with carry_pending the factors wait for more corrections (up to max_pending) before Sigma is swept
    return h->carry_pending ? EKF_OK : stream_flush(h, h->pending, nullptr);
}

int ekf_data_association(ekf_filter* h, const double* xy, int m, uint8_t* known, int32_t* assoc_out,
                         double* dmin_out, double* second_out, uint8_t* created_out) {
    if (!h || !known || m < 0 || (m > 0 && !xy)) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(h->device);
    if (h->engine != EKF_ENGINE_FUSED) {  // (the small engine's pending prediction rides along with the kernel below)
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    const int n = h->n;
    if (m == 0) return EKF_OK;
    int rc = ensure_m_cap(h, m);
    if (rc) return rc;
    unsigned char* slot;
    cudaEvent_t ev;
    rc = ring_acquire(h, &slot, &ev);
    if (rc) return rc;
    memcpy(slot, xy, sizeof(double) * 2 * m);
    memcpy(slot + sizeof(double) * 2 * m, known, n);
    int32_t* slot_i = reinterpret_cast<int32_t*>(slot + sizeof(double) * 2 * m + ((n + 15) & ~15));
    int known_count = 0;
    while (known_count < n && known[known_count]) ++known_count;  // leading-true prefix, ekf_slam.cpp:281-288
    slot_i[0] = m;
    slot_i[1] = known_count;
    // outputs: one pinned staging area, one synchronisation
    unsigned char* o = h->h_out;
    int32_t* o_assoc = reinterpret_cast<int32_t*>(o);
    double* o_dmin = reinterpret_cast<double*>(o + (((size_t)m * 4 + 15) & ~(size_t)15));
    double* o_second = o_dmin + m;
    uint8_t* o_created = reinterpret_cast<uint8_t*>(o_second + m);
    uint8_t* o_known = o_created + ((m + 15) & ~15);
    int* o_kc = reinterpret_cast<int*>(o_known + ((n + 15) & ~15));
    if (h->engine == EKF_ENGINE_FUSED) {
        // the kernel reads the slot and writes the log straight into the pinned areas (device mapping of both)
        double* tw = reinterpret_cast<double*>(slot_i + 4);
        tw[0] = h->pred_tw[0];
        tw[1] = h->pred_tw[1];
        FusedParams p = fused_params(h, kDoAssociation | (h->pred_pending ? kDoPredict : 0), m);
        h->pred_pending = false;
        p.twists = tw;
        p.xy = reinterpret_cast<const double*>(slot);
        p.known = slot + sizeof(double) * 2 * m;
        p.mcount = slot_i;
        p.assoc_out = o_assoc;
        p.dmin_out = o_dmin;
        p.second_out = o_second;
        p.created_out = o_created;
        rc = launch_fused(p, h->stream, h->device);
        CU(cudaEventRecord(ev, h->stream));
        h->launches += 1;
        h->pose_host_ok = rc == EKF_OK;
        if (rc) return rc;
        CU(cudaStreamSynchronize(h->stream));
        memcpy(o_known, slot + sizeof(double) * 2 * m, n);
    } else {
        CU(cudaMemcpyAsync(h->d_in, slot, sizeof(double) * 2 * m, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(h->d_flags, slot + sizeof(double) * 2 * m, n, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(h->d_known_count, slot_i + 1, sizeof(int), cudaMemcpyHostToDevice, h->stream));
        CU(cudaEventRecord(ev, h->stream));
        for (int j = 0; j < m; ++j) {
            k_large_assoc<<<h->assoc_blocks, 256, 0, h->stream>>>(h->d_sigma, h->ld, h->d_state, n, h->d_in, j,
                                                                   h->d_known_count, h->d_partials, h->d_done, h->d_cmd,
                                                                   h->d_assoc, h->d_dmin, h->d_second, h->d_created);
            h->launches += 1;
            // the next measurement's distances need the corrected Sigma: one factor, applied at once
            rc = stream_correct(h, h->d_state, h->d_cmd, 0, 0.0, 0.0);
            if (rc) return rc;
            rc = stream_flush(h, 1, h->d_cmd);
            if (rc) return rc;
        }
        CU(cudaMemcpyAsync(o_assoc, h->d_assoc, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(o_dmin, h->d_dmin, sizeof(double) * m, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(o_second, h->d_second, sizeof(double) * m, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(o_created, h->d_created, m, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(o_kc, h->d_known_count, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    if (assoc_out) memcpy(assoc_out, o_assoc, sizeof(int32_t) * m);
    if (dmin_out) memcpy(dmin_out, o_dmin, sizeof(double) * m);
    if (second_out) memcpy(second_out, o_second, sizeof(double) * m);
    if (created_out) memcpy(created_out, o_created, m);
    if (h->engine == EKF_ENGINE_FUSED) {
        memcpy(known, o_known, n);
    } else {
        for (int i = known_count; i < *o_kc && i < n; ++i) known[i] = 1;
    }
    if (h->assoc_log) {  // the structured counterpart of the reference's print stream (ekf_slam.cpp:290-329)
        for (int j = 0; j < m; ++j)
            fprintf(h->assoc_log, "%llu,%d,%.17g,%.17g,%d,%.17g,%.17g,%d\n", (unsigned long long)h->assoc_calls, j, xy[2 * j],
                    xy[2 * j + 1], (int)o_assoc[j], o_dmin[j], o_second[j], (int)o_created[j]);
        fflush(h->assoc_log);
    }
    h->assoc_calls += 1;
    return EKF_OK;
}

// Association log: a CSV file with one line per measurement handed to data_association(),
//   call,index,x,y,landmark (-1 = dropped),min_distance,runner_up,created
// (what the reference only prints, ekf_slam.cpp:290-329).  path = NULL closes the log.
int ekf_association_log_open(ekf_filter* h, const char* path) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    if (h->assoc_log) fclose(h->assoc_log);
    h->assoc_log = nullptr;
    if (!path) return EKF_OK;
    h->assoc_log = fopen(path, "w");
    if (!h->assoc_log) return fail(EKF_ERR_INVALID, "cannot open %s", path);
    fprintf(h->assoc_log, "call,index,x,y,landmark,min_distance,runner_up,created\n");
    return EKF_OK;
}

int ekf_maha(ekf_filter* h, double mx, double my, int landmark, double* d_out) {
    if (!h || !d_out || landmark < 0 || landmark >= h->n) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    k_maha_one<<<1, 1, 0, h->stream>>>(h->d_sigma, h->ld, h->d_state, landmark, mx, my, h->d_scalar);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(d_out, h->d_scalar, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}

int ekf_get_state(ekf_filter* h, double* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    CU(cudaMemcpyAsync(out, h->d_state, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_set_state(ekf_filter* h, const double* in) {
    if (!h || !in) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    h->pose_host_ok = false;
    CU(cudaMemcpyAsync(h->d_state, in, sizeof(double) * h->N, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_get_pose(ekf_filter* h, double* out3) {
    if (!h || !out3) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    if (h->engine == EKF_ENGINE_FUSED && h->pose_host_ok && !h->external) {
        CU(cudaStreamSynchronize(h->stream));  // the last kernel left the pose in pinned memory
        out3[0] = h->h_pose[0];
        out3[1] = h->h_pose[1];
        out3[2] = h->h_pose[2];
        return EKF_OK;
    }
    CU(cudaMemcpyAsync(out3, h->d_state, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_get_landmarks(ekf_filter* h, double* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    CU(cudaMemcpyAsync(out, h->d_state + 3, sizeof(double) * 2 * h->n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_get_sigma(ekf_filter* h, double* out, int64_t ld) {
    if (!h || !out || ld < h->N) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    CU(cudaMemcpy2DAsync(out, sizeof(double) * ld, h->d_sigma, sizeof(double) * h->ld, sizeof(double) * h->N, h->N,
                         cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
// Selected rows of Sigma (each N doubles, row stride ld in `out`) and its diagonal: the parity checks of maps whose
// whole covariance does not fit the host comfortably (n = 40,000: 51 GB) read these instead of ekf_get_sigma.
int ekf_get_sigma_rows(ekf_filter* h, const int64_t* rows, int count, double* out, int64_t ld) {
    if (!h || count < 0 || (count > 0 && (!rows || !out)) || ld < h->N) return fail(EKF_ERR_INVALID, "invalid argument");
    for (int k = 0; k < count; ++k)
        if (rows[k] < 0 || rows[k] >= h->N) return fail(EKF_ERR_INVALID, "row %lld out of range", (long long)rows[k]);
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    for (int k = 0; k < count; ++k)
        CU(cudaMemcpyAsync(out + (size_t)k * ld, h->d_sigma + (size_t)rows[k] * h->ld, sizeof(double) * h->N,
                           cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_get_sigma_diag(ekf_filter* h, double* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    CU(cudaMemcpy2DAsync(out, sizeof(double), h->d_sigma, sizeof(double) * (h->ld + 1), sizeof(double), h->N,
                         cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_set_sigma(ekf_filter* h, const double* in, int64_t ld) {
    if (!h || !in || ld < h->N) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    CU(cudaMemcpy2DAsync(h->d_sigma, sizeof(double) * h->ld, in, sizeof(double) * ld, sizeof(double) * h->N, h->N,
                         cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_get_init_flag(ekf_filter* h, int* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    int32_t v = 0;
    CU(cudaMemcpyAsync(&v, h->d_init_flag, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    *out = v;
    return EKF_OK;
}
int ekf_set_init_flag(ekf_filter* h, int v) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    const int32_t f = v ? 1 : 0;
    CU(cudaMemcpyAsync(h->d_init_flag, &f, sizeof(f), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->init_flag_host = f;
    return EKF_OK;
}
int ekf_update_count(ekf_filter* h, uint64_t* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, h->d_nupd, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    *out = v;
    return EKF_OK;
}
int ekf_sync(ekf_filter* h) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    CU(cudaStreamSynchronize(h->stream));
    return EKF_OK;
}
int ekf_device_pointers(ekf_filter* h, void** sigma, int64_t* ld, void** state) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    {
        DeviceGuard g(h->device);
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    if (sigma) *sigma = h->d_sigma;
    if (ld) *ld = h->ld;
    if (state) *state = h->d_state;
    h->external = true;
    return EKF_OK;
}
// How many corrections the streamed engine may accumulate before it sweeps Sigma (1..kMaxPending = 20, default 14).  The result
// is bit-identical for every setting; 1 reproduces the reference's schedule of one full pass per correction.
int ekf_set_max_pending(ekf_filter* h, int max_pending) {
    if (!h || max_pending < 1 || max_pending > kMaxPending) return fail(EKF_ERR_INVALID, "max_pending must be 1..%d", kMaxPending);
    h->max_pending = max_pending;
    if (h->pending >= max_pending) {
        DeviceGuard g(h->device);
        return stream_settle(h);
    }
    return EKF_OK;
}
// 1 (default): factor pairs may stay pending across prediction() and measurement() calls, so that every sweep of the
// streamed engine carries max_pending corrections; 0: Sigma is brought up to date at the end of every measurement()
// (then the delayed application is bit-identical to one sweep per correction).  Either way every verb that reads
// Sigma settles it first.
int ekf_set_carry_pending(ekf_filter* h, int carry) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    h->carry_pending = carry ? 1 : 0;
    if (!h->carry_pending) {
        DeviceGuard g(h->device);
        return stream_settle(h);
    }
    return EKF_OK;
}
int ekf_sweep_count(ekf_filter* h, uint64_t* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    *out = h->sweeps;
    return EKF_OK;
}
int ekf_launch_count(ekf_filter* h, uint64_t* out) {
    if (!h || !out) return fail(EKF_ERR_INVALID, "null argument");
    *out = h->launches;
    return EKF_OK;
}
// CUDA-event stopwatch on the handle's own stream (torch.cuda.Event only sees torch's streams).
int ekf_timer_start(ekf_filter* h) {
    if (!h) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    {
        int rc_ = settle_prediction(h);
        if (rc_) return rc_;
    }
    if (!h->t0) {
        CU(cudaEventCreate(&h->t0));
        CU(cudaEventCreate(&h->t1));
    }
    CU(cudaEventRecord(h->t0, h->stream));
    return EKF_OK;
}
int ekf_timer_stop(ekf_filter* h, float* ms_out) {
    if (!h || !ms_out || !h->t0) return fail(EKF_ERR_INVALID, "timer not started");
    DeviceGuard g(h->device);
    {
        int rc_ = stream_settle(h);
        if (rc_) return rc_;
    }
    CU(cudaEventRecord(h->t1, h->stream));
    CU(cudaEventSynchronize(h->t1));
    CU(cudaEventElapsedTime(ms_out, h->t0, h->t1));
    return EKF_OK;
}

}  // extern "C"

// ======================================================================================= batch
// Sigma layout of a batch: register tile (n = 20, ekf_fused_tile.cuh), symmetric staircase (other n <= 64,
// ekf_fused_sym.cuh), or dense N x ld rows per filter in HBM (64 < n <= 1,024, ekf_batch_wide.cuh).
enum class Layout { Tile, Stair, Wide };

struct ekf_batch {
    long long B = 0;
    int n = 0, N = 0, device = 0, sm_count = 0;
    Layout layout = Layout::Stair;
    int sig_stride = 0, st_stride = 0;  // doubles per filter in d_sigma and d_state
    int st_len = 0;      // doubles per filter in the state array of a checkpoint
    long long ld = 0;    // wide: row stride of a filter's Sigma
    int grid = 0;        // wide: CTAs of the step kernel (each owns a set of factor slots)
    cudaStream_t stream = nullptr;       // compute
    cudaStream_t copy_stream = nullptr;  // H2D of the next step's inputs
    cudaStream_t out_stream = nullptr;   // D2H of results
    uint64_t launches = 0;
    double* d_sigma = nullptr;  // [B][sig_stride]: staircase (ekf_fused_sym.cuh), tile, or dense N x ld (wide)
    double* d_dense = nullptr;  // N x N scratch of ekf_batch_get_sigma
    double* d_state = nullptr;
    int32_t* d_init_flag = nullptr;
    uint8_t* d_known = nullptr;
    unsigned long long* d_nupd = nullptr;
    unsigned long long* d_sweeps = nullptr;  // wide: passes over a filter's Sigma, summed over the batch
    double2* d_wK = nullptr;                 // wide: [grid][kWidePending * ld + 16] factor slots
    double2* d_wW = nullptr;
    // double-buffered device inputs
    int m_cap = 0;
    double* d_twists[2] = {nullptr, nullptr};
    double* d_xy[2] = {nullptr, nullptr};
    uint8_t* d_vis[2] = {nullptr, nullptr};
    int32_t* d_count[2] = {nullptr, nullptr};  // [B + 1]: per-filter counts, or CSR offsets of the marker list
    int32_t* d_assoc = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr};
    cudaEvent_t ev_consumed[2] = {nullptr, nullptr};
    cudaEvent_t ev_step = nullptr;
    cudaEvent_t ev_out = nullptr;
    int slot = 0;
    double* d_poses = nullptr;
    double* d_acc4 = nullptr;
    double* d_truth = nullptr;
    // consistency read-out (ekf_batch_consistency.cuh), allocated on first use
    int cons_grid = 0;
    double* d_cons_part = nullptr;      // [cons_grid][8] per-CTA partials
    unsigned int* d_cons_done = nullptr;
    double* d_marg_pose = nullptr;      // [B][6]
    double* d_marg_lm = nullptr;        // [B][n][3]
    double* d_nees_lm = nullptr;        // landmark truth of ekf_batch_nees, lm_cap doubles
    long long lm_cap = 0;
    double* d_nees_pf = nullptr;        // [B][3]
    double* d_nees_out = nullptr;       // [8]
    // NIS (ekf_batch_set_nis): per-filter accumulators, allocated and zeroed on first use; read-out buffers
    bool nis_on = false;
    double* d_nis = nullptr;            // [B][4] = {sum NIS, sum NIS^2, #scored, #non-finite}
    int nis_grid = 0;
    double* d_nis_part = nullptr;       // [nis_grid][4] per-CTA partials of k_batch_nis
    unsigned int* d_nis_done = nullptr;
    double* d_nis_pf = nullptr;         // [B][4] host read-out staging
    double* d_nis_out = nullptr;        // [4]
    cudaEvent_t t0 = nullptr, t1[3] = {nullptr, nullptr, nullptr};
};

namespace {

int free_batch(ekf_batch* b) {
    if (!b) return EKF_OK;
    DeviceGuard g(b->device);
    cudaDeviceSynchronize();
    cudaFree(b->d_sigma);
    cudaFree(b->d_dense);
    if (b->layout != Layout::Tile) cudaFree(b->d_state);  // tile: the state lives inside the filter's block of d_sigma
    cudaFree(b->d_init_flag);
    cudaFree(b->d_known);
    cudaFree(b->d_nupd);
    cudaFree(b->d_sweeps);
    cudaFree(b->d_wK);
    cudaFree(b->d_wW);
    for (int s = 0; s < 2; ++s) {
        cudaFree(b->d_twists[s]);
        cudaFree(b->d_xy[s]);
        cudaFree(b->d_vis[s]);
        cudaFree(b->d_count[s]);
        if (b->ev_copied[s]) cudaEventDestroy(b->ev_copied[s]);
        if (b->ev_consumed[s]) cudaEventDestroy(b->ev_consumed[s]);
    }
    cudaFree(b->d_assoc);
    cudaFree(b->d_poses);
    cudaFree(b->d_acc4);
    cudaFree(b->d_truth);
    cudaFree(b->d_cons_part);
    cudaFree(b->d_cons_done);
    cudaFree(b->d_marg_pose);
    cudaFree(b->d_marg_lm);
    cudaFree(b->d_nees_lm);
    cudaFree(b->d_nees_pf);
    cudaFree(b->d_nees_out);
    cudaFree(b->d_nis);
    cudaFree(b->d_nis_part);
    cudaFree(b->d_nis_done);
    cudaFree(b->d_nis_pf);
    cudaFree(b->d_nis_out);
    if (b->ev_step) cudaEventDestroy(b->ev_step);
    if (b->ev_out) cudaEventDestroy(b->ev_out);
    if (b->t0) cudaEventDestroy(b->t0);
    for (int i = 0; i < 3; ++i)
        if (b->t1[i]) cudaEventDestroy(b->t1[i]);
    if (b->stream) cudaStreamDestroy(b->stream);
    if (b->copy_stream) cudaStreamDestroy(b->copy_stream);
    if (b->out_stream) cudaStreamDestroy(b->out_stream);
    cudaGetLastError();
    delete b;
    return EKF_OK;
}

int batch_ensure_xy(ekf_batch* b, int m_max) {
    const int need = std::max(b->n, m_max);
    if (need <= b->m_cap) return EKF_OK;
    CU(cudaDeviceSynchronize());
    for (int s = 0; s < 2; ++s) {
        cudaFree(b->d_xy[s]);
        b->d_xy[s] = nullptr;
        CU(cudaMalloc(&b->d_xy[s], sizeof(double) * 2 * (size_t)need * b->B));
    }
    cudaFree(b->d_assoc);
    b->d_assoc = nullptr;
    CU(cudaMalloc(&b->d_assoc, sizeof(int32_t) * (size_t)need * b->B));
    b->m_cap = need;
    return EKF_OK;
}

// Layout and strides of a batch of n-landmark filters.
void batch_geometry(ekf_batch* b) {
    if (b->n == tile::kNL) {
        // one block per filter holds Sigma (fragment layout) and the state, so that one bulk copy stages it; a
        // checkpoint keeps the state as its own compact array as well
        b->layout = Layout::Tile;
        b->sig_stride = b->st_stride = tile::kStride;
        b->st_len = tile::kStLen;
    } else if (b->n <= kFusedMaxN) {
        b->layout = Layout::Stair;
        b->sig_stride = sym_sig_stride(b->N);
        b->st_stride = b->st_len = sym_st_stride(b->N);
    } else {  // the streamed engine's layout: row-major N x ld, ld = N rounded up to 16 doubles
        b->layout = Layout::Wide;
        b->ld = fused_round16(b->N);
        b->sig_stride = b->N * (int)b->ld;
        b->st_stride = b->st_len = (int)b->ld;
    }
}

// Buffers and initial state of a new batch; on failure the caller frees the half-made handle.
int alloc_batch(ekf_batch* b) {
    const long long B = b->B;
    const int n = b->n;
    CU(cudaDeviceGetAttribute(&b->sm_count, cudaDevAttrMultiProcessorCount, b->device));
    CU(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&b->out_stream, cudaStreamNonBlocking));
    CU(cudaMalloc(&b->d_sigma, sizeof(double) * (size_t)b->sig_stride * B));
    if (b->layout == Layout::Tile)
        b->d_state = b->d_sigma + tile::kStOff;
    else
        CU(cudaMalloc(&b->d_state, sizeof(double) * (size_t)b->st_stride * B));
    CU(cudaMalloc(&b->d_init_flag, sizeof(int32_t) * (size_t)B));
    CU(cudaMalloc(&b->d_known, (size_t)n * B));
    CU(cudaMalloc(&b->d_nupd, sizeof(unsigned long long)));
    CU(cudaMalloc(&b->d_poses, sizeof(double) * 3 * (size_t)B));
    CU(cudaMalloc(&b->d_acc4, sizeof(double) * 4));
    CU(cudaMalloc(&b->d_truth, sizeof(double) * 3 * (size_t)B));
    for (int s = 0; s < 2; ++s) {
        CU(cudaMalloc(&b->d_twists[s], sizeof(double) * 2 * (size_t)B));
        CU(cudaMalloc(&b->d_vis[s], (size_t)n * B));
        CU(cudaMalloc(&b->d_count[s], sizeof(int32_t) * ((size_t)B + 1)));
        CU(cudaEventCreateWithFlags(&b->ev_copied[s], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&b->ev_consumed[s], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&b->ev_step, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&b->ev_out, cudaEventDisableTiming));
    CU(cudaMemsetAsync(b->d_known, 0, (size_t)n * B, b->stream));
    CU(cudaMemsetAsync(b->d_nupd, 0, sizeof(unsigned long long), b->stream));
    switch (b->layout) {
        case Layout::Tile:
            tile::k_fused_tile_init<<<(unsigned)B, 128, 0, b->stream>>>(b->d_sigma, b->d_init_flag, B);
            break;
        case Layout::Stair:
            k_fused_sym_init<<<(unsigned)B, 128, 0, b->stream>>>(b->d_sigma, b->d_state, b->d_init_flag, B, b->N,
                                                                 b->sig_stride, b->st_stride);
            break;
        case Layout::Wide: {
            b->grid = (int)std::min<long long>(B, std::max(b->sm_count, 1));
            const size_t slots = (size_t)b->grid * ((size_t)kWidePending * b->ld + 16);
            CU(cudaMalloc(&b->d_wK, sizeof(double2) * slots));
            CU(cudaMalloc(&b->d_wW, sizeof(double2) * slots));
            CU(cudaMalloc(&b->d_sweeps, sizeof(unsigned long long)));
            CU(cudaMemsetAsync(b->d_wK, 0, sizeof(double2) * slots, b->stream));
            CU(cudaMemsetAsync(b->d_wW, 0, sizeof(double2) * slots, b->stream));
            CU(cudaMemsetAsync(b->d_sweeps, 0, sizeof(unsigned long long), b->stream));
            CU(cudaMemsetAsync(b->d_sigma, 0, sizeof(double) * (size_t)b->sig_stride * B, b->stream));
            CU(cudaMemsetAsync(b->d_state, 0, sizeof(double) * (size_t)b->st_stride * B, b->stream));
            CU(cudaMemsetAsync(b->d_init_flag, 0, sizeof(int32_t) * (size_t)B, b->stream));
            const long long diag = B * (b->N - 3);
            k_init_sigma<<<(unsigned)((diag + 255) / 256), 256, 0, b->stream>>>(b->d_sigma, B, b->N, b->ld, b->sig_stride);
            break;
        }
    }
    b->launches += 1;
    CU(cudaGetLastError());
    int rc = batch_ensure_xy(b, n);
    if (rc) return rc;
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}

// One step of a wide batch: dense readings (offsets == nullptr) or the marker list.
int launch_wide(ekf_batch* b, const double* twists, const double* xy, const uint8_t* vis, const int32_t* offsets,
                long long total) {
    WideParams p;
    memset(&p, 0, sizeof(p));
    p.sigma = b->d_sigma;
    p.state = b->d_state;
    p.init_flag = b->d_init_flag;
    p.n_updates = b->d_nupd;
    p.n_sweeps = b->d_sweeps;
    p.Kp = b->d_wK;
    p.Wp = b->d_wW;
    p.twists = twists;
    p.xy = xy;
    p.vis = vis;
    p.offsets = offsets;
    p.sparse_total = total;
    p.B = b->B;
    p.ld = b->ld;
    p.slot_stride = (long long)kWidePending * b->ld + 16;
    p.n = b->n;
    p.N = b->N;
    p.st_stride = b->st_stride;
    p.nis = b->nis_on ? b->d_nis : nullptr;
    if (p.nis)
        CU(launch_wide_step<true>(p, b->grid, b->stream, b->device));
    else
        CU(launch_wide_step<false>(p, b->grid, b->stream, b->device));
    return EKF_OK;
}

// One step of the whole batch in the kernel of its layout, counted as one launch; with NIS on, the NIS variant of that
// kernel (ekf_batch_set_nis).  `mode` as in FusedParams; `vis`
// holds the visible flags, or the marker ids with kSparseReadings; `cnt` the marker list's CSR offsets, or the
// per-filter measurement counts of unknown association.
int batch_launch(ekf_batch* b, int mode, int m_max, const double* tw, const double* xy, const uint8_t* vis,
                 const int32_t* cnt, int32_t* assoc, long long total) {
    const bool association = (mode & kDoAssociation) != 0;
    int rc;
    if (b->layout == Layout::Wide) {
        if (association)
            return fail(EKF_ERR_UNSUPPORTED,
                        "unknown data association is not available for batches with n > %d landmarks", kFusedMaxN);
        rc = launch_wide(b, tw, xy, vis, cnt, total);
    } else {
        FusedParams p;
        memset(&p, 0, sizeof(p));
        p.sigma = b->d_sigma;
        p.state = b->d_state;
        p.init_flag = b->d_init_flag;
        p.known = b->d_known;
        p.twists = tw;
        p.xy = xy;
        p.vis = vis;
        p.mcount = cnt;
        p.assoc_out = assoc;
        p.n_updates = b->d_nupd;
        p.B = b->B;
        p.n = b->n;
        p.m_max = m_max;
        p.mode = mode;
        p.sig_stride = b->sig_stride;
        p.st_stride = b->st_stride;
        p.sparse_total = total;
        p.nis = b->nis_on ? b->d_nis : nullptr;
        if (b->layout == Layout::Stair)
            rc = launch_fused_staircase(p, b->stream, b->device);
        else if (association)
            rc = p.nis ? launch_fused_tile<true, true>(p, b->stream, b->device, b->sm_count)
                       : launch_fused_tile<true, false>(p, b->stream, b->device, b->sm_count);
        else
            rc = p.nis ? launch_fused_tile<false, true>(p, b->stream, b->device, b->sm_count)
                       : launch_fused_tile<false, false>(p, b->stream, b->device, b->sm_count);
    }
    b->launches += 1;
    return rc;
}

struct HostCopy {
    void* dst;
    const void* src;
    size_t bytes;  // 0: skipped
};

// A step fed from host memory through the double-buffered device inputs: `copies` fill input slot b->slot on the copy
// stream once the step that last read that slot has finished, and step() is enqueued on the compute stream behind
// them.  The next host-fed step uses the other slot.
template <class Step>
int batch_host_step(ekf_batch* b, std::initializer_list<HostCopy> copies, Step step) {
    const int s = b->slot;
    b->slot ^= 1;
    CU(cudaStreamWaitEvent(b->copy_stream, b->ev_consumed[s], 0));
    for (const HostCopy& c : copies)
        if (c.bytes) CU(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyHostToDevice, b->copy_stream));
    CU(cudaEventRecord(b->ev_copied[s], b->copy_stream));
    CU(cudaStreamWaitEvent(b->stream, b->ev_copied[s], 0));
    const int rc = step();
    if (rc) return rc;
    CU(cudaEventRecord(b->ev_consumed[s], b->stream));
    return EKF_OK;
}

// The marker list carries uint8_t landmark ids.
constexpr int kMarkerMaxN = 256;

// One launch of k_batch_consistency on the compute stream, in the batch's Sigma layout.  The grid is what fits the
// device at once (each warp walks filters w, w + warps, ...), fixed for the handle so that the reduction order is too.
template <class At>
int launch_consistency_at(ekf_batch* b, const ConsistencyParams& p, At at) {
    if (!b->cons_grid) {
        int per_sm = 0;
        CU(kernel_setup<k_batch_consistency<At>>(b->device, kConsWarps * 32, 0, false, &per_sm));
        const long long resident = (long long)std::max(b->sm_count, 1) * std::max(per_sm, 1);
        const int grid = (int)std::min<long long>((b->B + kConsWarps - 1) / kConsWarps, resident);
        CU(cudaMalloc(&b->d_cons_part, sizeof(double) * 8 * (size_t)grid));
        CU(cudaMalloc(&b->d_cons_done, sizeof(unsigned int)));
        CU(cudaMemsetAsync(b->d_cons_done, 0, sizeof(unsigned int), b->stream));
        b->cons_grid = grid;
    }
    ConsistencyParams q = p;
    q.partials = b->d_cons_part;
    q.done = b->d_cons_done;
    k_batch_consistency<At><<<b->cons_grid, kConsWarps * 32, 0, b->stream>>>(q, at);
    b->launches += 1;
    CU(cudaGetLastError());
    return EKF_OK;
}

int launch_consistency(ekf_batch* b, const double* truth, const double* lm_truth, long long lm_stride,
                       double* per_filter, double* pose_cov, double* lm_cov, double* out8) {
    ConsistencyParams p;
    memset(&p, 0, sizeof(p));
    p.state = b->d_state;
    p.init_flag = b->d_init_flag;
    p.known = b->d_known;
    p.truth = truth;
    p.lm_truth = lm_truth;
    p.per_filter = per_filter;
    p.pose_cov = pose_cov;
    p.lm_cov = lm_cov;
    p.out8 = out8;
    p.B = b->B;
    p.st_stride = b->st_stride;
    p.lm_stride = lm_stride;
    p.n = b->n;
    if (b->layout == Layout::Wide) return launch_consistency_at(b, p, WideAt{b->d_sigma, b->sig_stride, b->ld});
    if (b->layout == Layout::Tile) return launch_consistency_at(b, p, TileAt{b->d_sigma});
    return launch_consistency_at(b, p, StairAt{b->d_sigma, b->sig_stride, b->N});
}

// One launch of k_batch_nis on the compute stream; the grid is fixed for the handle, so the reduction order is too.
int launch_nis(ekf_batch* b, double* per_filter, double* out4, int reset) {
    if (!b->nis_grid) {
        int per_sm = 0;
        CU(kernel_setup<k_batch_nis>(b->device, kConsWarps * 32, 0, false, &per_sm));
        const long long resident = (long long)std::max(b->sm_count, 1) * std::max(per_sm, 1);
        const int grid = (int)std::min<long long>((b->B + kConsWarps * 32 - 1) / (kConsWarps * 32), resident);
        CU(cudaMalloc(&b->d_nis_part, sizeof(double) * 4 * (size_t)grid));
        CU(cudaMalloc(&b->d_nis_done, sizeof(unsigned int)));
        CU(cudaMemsetAsync(b->d_nis_done, 0, sizeof(unsigned int), b->stream));
        b->nis_grid = grid;
    }
    k_batch_nis<<<b->nis_grid, kConsWarps * 32, 0, b->stream>>>(b->d_nis, b->B, per_filter, reset != 0, b->d_nis_part,
                                                              b->d_nis_done, out4);
    b->launches += 1;
    CU(cudaGetLastError());
    return EKF_OK;
}

int check_nis_args(ekf_batch* b, const double* out4) {
    if (!b || !out4) return fail(EKF_ERR_INVALID, "null argument");
    if (!b->d_nis) return fail(EKF_ERR_STATE, "NIS was never enabled on this batch (ekf_batch_set_nis)");
    return EKF_OK;
}

int check_nees_args(ekf_batch* b, const double* truth, int64_t lm_truth_stride, const double* out8) {
    if (!b || !truth || !out8) return fail(EKF_ERR_INVALID, "null argument");
    if (lm_truth_stride != 0 && lm_truth_stride != 2LL * b->n)
        return fail(EKF_ERR_INVALID, "lm_truth_stride must be 0 (shared landmark truth) or 2n = %d", 2 * b->n);
    return EKF_OK;
}

}  // namespace

extern "C" {

int ekf_batch_create(int64_t B, int n, int device, ekf_batch** out) {
    if (!out) return fail(EKF_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (B <= 0 || n <= 0) return fail(EKF_ERR_INVALID, "invalid batch shape");
    if (B > 0x7fffffffLL) return fail(EKF_ERR_INVALID, "batch too large");
    if (n > kWideMaxN)
        return fail(EKF_ERR_UNSUPPORTED,
                    "batched filters support n <= %d landmarks; for a larger map use one streamed filter per map, "
                    "ekf_create_ex(n, device, EKF_ENGINE_STREAM, &h)",
                    kWideMaxN);
    int rc = check_device(device);
    if (rc) return rc;
    DeviceGuard g(device);
    ekf_batch* b = new (std::nothrow) ekf_batch();
    if (!b) return fail(EKF_ERR_STATE, "out of host memory");
    b->B = B;
    b->n = n;
    b->N = 3 + 2 * n;
    b->device = device;
    batch_geometry(b);
    rc = alloc_batch(b);
    if (rc) {
        free_batch(b);
        return rc;
    }
    *out = b;
    return EKF_OK;
}

int ekf_batch_destroy(ekf_batch* b) { return free_batch(b); }
int64_t ekf_batch_size(const ekf_batch* b) { return b ? b->B : EKF_ERR_INVALID; }
int ekf_batch_engine(const ekf_batch* b) {
    return b ? (b->layout == Layout::Wide ? EKF_ENGINE_STREAM : EKF_ENGINE_FUSED) : EKF_ERR_INVALID;
}
int ekf_batch_sweep_count(ekf_batch* b, uint64_t* out) {
    if (!b || !out) return fail(EKF_ERR_INVALID, "null argument");
    *out = 0;
    if (b->layout != Layout::Wide) return EKF_OK;  // the on-chip engines never sweep a covariance in HBM
    DeviceGuard g(b->device);
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, b->d_sweeps, sizeof(v), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    *out = v;
    return EKF_OK;
}
void* ekf_batch_stream(ekf_batch* b) { return b ? (void*)b->stream : nullptr; }

int ekf_batch_step_known_dev(ekf_batch* b, const double* d_twists, const double* d_xy, const uint8_t* d_visible) {
    if (!b || !d_twists || !d_xy || !d_visible) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    return batch_launch(b, kDoPredict | kDoMeasurement, 1, d_twists, d_xy, d_visible, nullptr, nullptr, 0);
}

int ekf_batch_step_unknown_dev(ekf_batch* b, const double* d_twists, const double* d_meas, const int32_t* d_count,
                               int m_max, int32_t* d_assoc_out) {
    if (!b || !d_twists || !d_meas || m_max <= 0) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(b->device);
    return batch_launch(b, kDoPredict | kDoAssociation, m_max, d_twists, d_meas, nullptr, d_count, d_assoc_out, 0);
}

int ekf_batch_step_known(ekf_batch* b, const double* twists, const double* xy, const uint8_t* visible) {
    if (!b || !twists || !xy || !visible) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B, n = (size_t)b->n;
    const int s = b->slot;
    return batch_host_step(b,
                           {{b->d_twists[s], twists, sizeof(double) * 2 * B},
                            {b->d_xy[s], xy, sizeof(double) * 2 * n * B},
                            {b->d_vis[s], visible, n * B}},
                           [&] {
                               return batch_launch(b, kDoPredict | kDoMeasurement, 1, b->d_twists[s], b->d_xy[s],
                                                   b->d_vis[s], nullptr, nullptr, 0);
                           });
}

int ekf_batch_step_known_sparse_dev(ekf_batch* b, const double* d_twists, const int32_t* d_offsets, const uint8_t* d_ids,
                                    const double* d_xy, int64_t total) {
    if (!b || !d_twists || !d_offsets || !d_ids || !d_xy || total < 0) return fail(EKF_ERR_INVALID, "invalid argument");
    if (b->n > kMarkerMaxN)
        return fail(EKF_ERR_UNSUPPORTED, "the marker list carries uint8 ids: n <= %d landmarks (use the dense arrays)",
                    kMarkerMaxN);
    DeviceGuard g(b->device);
    return batch_launch(b, kDoPredict | kDoMeasurement | kSparseReadings, 1, d_twists, d_xy, d_ids, d_offsets, nullptr,
                        total);
}

int ekf_batch_step_known_sparse(ekf_batch* b, const double* twists, const int32_t* offsets, const uint8_t* ids,
                                const double* xy, int64_t total) {
    if (!b || !twists || !offsets || total < 0 || (total > 0 && (!ids || !xy)))
        return fail(EKF_ERR_INVALID, "null argument");
    if (total > (int64_t)b->n * b->B) return fail(EKF_ERR_INVALID, "marker list longer than n markers per filter");
    if (b->n > kMarkerMaxN)
        return fail(EKF_ERR_UNSUPPORTED, "the marker list carries uint8 ids: n <= %d landmarks (use the dense arrays)",
                    kMarkerMaxN);
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B;
    const int s = b->slot;
    return batch_host_step(b,
                           {{b->d_twists[s], twists, sizeof(double) * 2 * B},
                            {b->d_count[s], offsets, sizeof(int32_t) * (B + 1)},
                            {b->d_vis[s], ids, (size_t)total},
                            {b->d_xy[s], xy, sizeof(double) * 2 * (size_t)total}},
                           [&] {
                               return batch_launch(b, kDoPredict | kDoMeasurement | kSparseReadings, 1, b->d_twists[s],
                                                   b->d_xy[s], b->d_vis[s], b->d_count[s], nullptr, total);
                           });
}

int ekf_batch_step_unknown(ekf_batch* b, const double* twists, const double* meas, const int32_t* count, int m_max,
                           int32_t* assoc_out) {
    if (!b || !twists || !meas || !count || m_max <= 0) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(b->device);
    int rc = batch_ensure_xy(b, m_max);
    if (rc) return rc;
    const size_t B = (size_t)b->B;
    const int s = b->slot;
    rc = batch_host_step(b,
                         {{b->d_twists[s], twists, sizeof(double) * 2 * B},
                          {b->d_xy[s], meas, sizeof(double) * 2 * m_max * B},
                          {b->d_count[s], count, sizeof(int32_t) * B}},
                         [&] {
                             return batch_launch(b, kDoPredict | kDoAssociation, m_max, b->d_twists[s], b->d_xy[s],
                                                 nullptr, b->d_count[s], assoc_out ? b->d_assoc : nullptr, 0);
                         });
    if (rc || !assoc_out) return rc;
    CU(cudaMemcpyAsync(assoc_out, b->d_assoc, sizeof(int32_t) * m_max * B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}

int ekf_batch_get_poses_async(ekf_batch* b, double* pinned_out) {
    if (!b || !pinned_out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    // gather on the compute stream (ordered after the step), copy out on the output stream
    CU(cudaStreamWaitEvent(b->stream, b->ev_out, 0));  // previous read-back of d_poses must be done
    const long long total = 3 * b->B;
    k_gather_poses<<<(unsigned)((total + 255) / 256), 256, 0, b->stream>>>(b->d_state, b->B, b->st_stride, b->d_poses);
    b->launches += 1;
    CU(cudaGetLastError());
    CU(cudaEventRecord(b->ev_step, b->stream));
    CU(cudaStreamWaitEvent(b->out_stream, b->ev_step, 0));
    CU(cudaMemcpyAsync(pinned_out, b->d_poses, sizeof(double) * (size_t)total, cudaMemcpyDeviceToHost, b->out_stream));
    CU(cudaEventRecord(b->ev_out, b->out_stream));
    return EKF_OK;
}

int ekf_batch_get_poses(ekf_batch* b, double* out) {
    int rc = ekf_batch_get_poses_async(b, out);
    if (rc) return rc;
    DeviceGuard g(b->device);
    CU(cudaStreamSynchronize(b->out_stream));
    return EKF_OK;
}

int ekf_batch_get_states(ekf_batch* b, double* out) {
    if (!b || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    CU(cudaMemcpy2DAsync(out, sizeof(double) * b->N, b->d_state, sizeof(double) * b->st_stride, sizeof(double) * b->N,
                         (size_t)b->B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}

int ekf_batch_get_sigma(ekf_batch* b, int64_t filter, double* out, int64_t ld) {
    if (!b || !out || filter < 0 || filter >= b->B || ld < b->N) return fail(EKF_ERR_INVALID, "invalid argument");
    DeviceGuard g(b->device);
    const double* src = b->d_sigma + (size_t)filter * b->sig_stride;
    long long src_ld = b->ld;
    if (b->layout != Layout::Wide) {  // the on-chip layouts: expand the filter's copy to dense N x N first
        if (!b->d_dense) CU(cudaMalloc(&b->d_dense, sizeof(double) * (size_t)b->N * b->N));
        const int blocks = (b->N * b->N + 255) / 256;
        if (b->layout == Layout::Tile)
            tile::k_fused_tile_unpack<<<blocks, 256, 0, b->stream>>>(src, b->d_dense);
        else
            k_fused_sym_unpack<<<blocks, 256, 0, b->stream>>>(src, b->d_dense, b->N);
        CU(cudaGetLastError());
        src = b->d_dense;
        src_ld = b->N;
    }
    CU(cudaMemcpy2DAsync(out, sizeof(double) * ld, src, sizeof(double) * src_ld, sizeof(double) * b->N, b->N,
                         cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}

int ekf_batch_get_known(ekf_batch* b, uint8_t* out) {
    if (!b || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    CU(cudaMemcpyAsync(out, b->d_known, (size_t)b->n * b->B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}
// Checkpoint / resume of the whole batch: the arrays exactly as the engine keeps them (Sigma in the engine's layout:
// packed symmetric, tile or dense N x ld; per-filter strides as reported by ekf_batch_checkpoint_size).  No conversion, so a restored batch continues
// bit-identically.
int ekf_batch_checkpoint_size(ekf_batch* b, int64_t* sigma_doubles, int64_t* state_doubles) {
    if (!b) return fail(EKF_ERR_INVALID, "null handle");
    if (sigma_doubles) *sigma_doubles = (int64_t)b->sig_stride * b->B;
    if (state_doubles) *state_doubles = (int64_t)b->st_len * b->B;
    return EKF_OK;
}
int ekf_batch_export(ekf_batch* b, double* sigma, double* state, int32_t* init_flag, uint8_t* known, uint64_t* updates) {
    if (!b || !sigma || !state || !init_flag || !known) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B;
    CU(cudaStreamSynchronize(b->copy_stream));
    CU(cudaMemcpyAsync(sigma, b->d_sigma, sizeof(double) * b->sig_stride * B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaMemcpy2DAsync(state, sizeof(double) * b->st_len, b->d_state, sizeof(double) * b->st_stride,
                         sizeof(double) * b->st_len, B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaMemcpyAsync(init_flag, b->d_init_flag, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaMemcpyAsync(known, b->d_known, (size_t)b->n * B, cudaMemcpyDeviceToHost, b->stream));
    unsigned long long u = 0;
    CU(cudaMemcpyAsync(&u, b->d_nupd, sizeof(u), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    if (updates) *updates = (uint64_t)u;
    return EKF_OK;
}
int ekf_batch_import(ekf_batch* b, const double* sigma, const double* state, const int32_t* init_flag,
                     const uint8_t* known, uint64_t updates) {
    if (!b || !sigma || !state || !init_flag || !known) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B;
    CU(cudaStreamSynchronize(b->copy_stream));
    CU(cudaStreamSynchronize(b->out_stream));
    CU(cudaMemcpyAsync(b->d_sigma, sigma, sizeof(double) * b->sig_stride * B, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpy2DAsync(b->d_state, sizeof(double) * b->st_stride, state, sizeof(double) * b->st_len,
                         sizeof(double) * b->st_len, B, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(b->d_init_flag, init_flag, sizeof(int32_t) * B, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(b->d_known, known, (size_t)b->n * B, cudaMemcpyHostToDevice, b->stream));
    const unsigned long long u = (unsigned long long)updates;
    CU(cudaMemcpyAsync(b->d_nupd, &u, sizeof(u), cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}
int ekf_batch_set_known(ekf_batch* b, const uint8_t* in) {
    if (!b || !in) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    CU(cudaMemcpyAsync(b->d_known, in, (size_t)b->n * b->B, cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}
int ekf_batch_update_count(ekf_batch* b, uint64_t* out) {
    if (!b || !out) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, b->d_nupd, sizeof(v), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    *out = v;
    return EKF_OK;
}
int ekf_batch_pose_error(ekf_batch* b, const double* truth, double* out4) {
    if (!b || !truth || !out4) return fail(EKF_ERR_INVALID, "null argument");
    DeviceGuard g(b->device);
    CU(cudaMemcpyAsync(b->d_truth, truth, sizeof(double) * 3 * (size_t)b->B, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemsetAsync(b->d_acc4, 0, sizeof(double) * 4, b->stream));
    const int blocks = (int)std::min<long long>((b->B + 255) / 256, 1184);
    k_pose_error<<<blocks, 256, 0, b->stream>>>(b->d_state, b->B, b->st_stride, b->d_truth, b->d_acc4);
    b->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out4, b->d_acc4, sizeof(double) * 4, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    out4[3] = (double)b->B;
    return EKF_OK;
}
int ekf_batch_get_marginals(ekf_batch* b, double* pose_cov, double* lm_cov) {
    if (!b) return fail(EKF_ERR_INVALID, "null handle");
    if (!pose_cov && !lm_cov) return EKF_OK;
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B;
    if (pose_cov && !b->d_marg_pose) CU(cudaMalloc(&b->d_marg_pose, sizeof(double) * 6 * B));
    if (lm_cov && !b->d_marg_lm) CU(cudaMalloc(&b->d_marg_lm, sizeof(double) * 3 * (size_t)b->n * B));
    int rc = launch_consistency(b, nullptr, nullptr, 0, nullptr, pose_cov ? b->d_marg_pose : nullptr,
                                lm_cov ? b->d_marg_lm : nullptr, nullptr);
    if (rc) return rc;
    if (pose_cov) CU(cudaMemcpyAsync(pose_cov, b->d_marg_pose, sizeof(double) * 6 * B, cudaMemcpyDeviceToHost, b->stream));
    if (lm_cov)
        CU(cudaMemcpyAsync(lm_cov, b->d_marg_lm, sizeof(double) * 3 * (size_t)b->n * B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}
int ekf_batch_nees(ekf_batch* b, const double* truth, const double* lm_truth, int64_t lm_truth_stride, double* per_filter,
                   double* out8) {
    int rc = check_nees_args(b, truth, lm_truth_stride, out8);
    if (rc) return rc;
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B;
    const long long lm_len = lm_truth ? 2LL * b->n * (lm_truth_stride ? b->B : 1) : 0;
    if (lm_len > b->lm_cap) {
        CU(cudaStreamSynchronize(b->stream));
        cudaFree(b->d_nees_lm);
        b->d_nees_lm = nullptr;
        b->lm_cap = 0;
        CU(cudaMalloc(&b->d_nees_lm, sizeof(double) * (size_t)lm_len));
        b->lm_cap = lm_len;
    }
    if (per_filter && !b->d_nees_pf) CU(cudaMalloc(&b->d_nees_pf, sizeof(double) * 3 * B));
    if (!b->d_nees_out) CU(cudaMalloc(&b->d_nees_out, sizeof(double) * 8));
    CU(cudaMemcpyAsync(b->d_truth, truth, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, b->stream));
    if (lm_truth)
        CU(cudaMemcpyAsync(b->d_nees_lm, lm_truth, sizeof(double) * (size_t)lm_len, cudaMemcpyHostToDevice, b->stream));
    rc = launch_consistency(b, b->d_truth, lm_truth ? b->d_nees_lm : nullptr, lm_truth_stride,
                            per_filter ? b->d_nees_pf : nullptr, nullptr, nullptr, b->d_nees_out);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out8, b->d_nees_out, sizeof(double) * 8, cudaMemcpyDeviceToHost, b->stream));
    if (per_filter) CU(cudaMemcpyAsync(per_filter, b->d_nees_pf, sizeof(double) * 3 * B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}
int ekf_batch_nees_dev(ekf_batch* b, const double* d_truth, const double* d_lm_truth, int64_t lm_truth_stride,
                       double* d_per_filter, double* d_out8) {
    int rc = check_nees_args(b, d_truth, lm_truth_stride, d_out8);
    if (rc) return rc;
    DeviceGuard g(b->device);
    return launch_consistency(b, d_truth, d_lm_truth, lm_truth_stride, d_per_filter, nullptr, nullptr, d_out8);
}
int ekf_batch_set_nis(ekf_batch* b, int on) {
    if (!b) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(b->device);
    if (on && !b->d_nis) {
        CU(cudaMalloc(&b->d_nis, sizeof(double) * 4 * (size_t)b->B));
        CU(cudaMemsetAsync(b->d_nis, 0, sizeof(double) * 4 * (size_t)b->B, b->stream));
    }
    b->nis_on = on != 0;
    return EKF_OK;
}
int ekf_batch_nis(ekf_batch* b, double* per_filter, double* out4, int reset) {
    int rc = check_nis_args(b, out4);
    if (rc) return rc;
    DeviceGuard g(b->device);
    const size_t B = (size_t)b->B;
    if (per_filter && !b->d_nis_pf) CU(cudaMalloc(&b->d_nis_pf, sizeof(double) * 4 * B));
    if (!b->d_nis_out) CU(cudaMalloc(&b->d_nis_out, sizeof(double) * 4));
    rc = launch_nis(b, per_filter ? b->d_nis_pf : nullptr, b->d_nis_out, reset);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out4, b->d_nis_out, sizeof(double) * 4, cudaMemcpyDeviceToHost, b->stream));
    if (per_filter) CU(cudaMemcpyAsync(per_filter, b->d_nis_pf, sizeof(double) * 4 * B, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return EKF_OK;
}
int ekf_batch_nis_dev(ekf_batch* b, double* d_per_filter, double* d_out4, int reset) {
    int rc = check_nis_args(b, d_out4);
    if (rc) return rc;
    DeviceGuard g(b->device);
    return launch_nis(b, d_per_filter, d_out4, reset);
}
int ekf_batch_sync(ekf_batch* b) {
    if (!b) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(b->device);
    CU(cudaStreamSynchronize(b->copy_stream));
    CU(cudaStreamSynchronize(b->stream));
    CU(cudaStreamSynchronize(b->out_stream));
    return EKF_OK;
}
int ekf_batch_device_pointers(ekf_batch* b, void** sigma, int64_t* sigma_stride, void** state, int64_t* state_stride) {
    if (!b) return fail(EKF_ERR_INVALID, "null handle");
    if (sigma) *sigma = b->d_sigma;
    if (sigma_stride) *sigma_stride = b->sig_stride;
    if (state) *state = b->d_state;
    if (state_stride) *state_stride = b->st_stride;
    return EKF_OK;
}
// Stopwatch over all three of the handle's streams: start is recorded on the (idle) compute stream, stop on
// compute, copy and output streams; the elapsed time is the latest of the three.
int ekf_batch_timer_start(ekf_batch* b) {
    if (!b) return fail(EKF_ERR_INVALID, "null handle");
    DeviceGuard g(b->device);
    if (!b->t0) {
        CU(cudaEventCreate(&b->t0));
        for (int i = 0; i < 3; ++i) CU(cudaEventCreate(&b->t1[i]));
    }
    CU(cudaEventRecord(b->t0, b->stream));
    return EKF_OK;
}
int ekf_batch_timer_stop(ekf_batch* b, float* ms_out) {
    if (!b || !ms_out || !b->t0) return fail(EKF_ERR_INVALID, "timer not started");
    DeviceGuard g(b->device);
    cudaStream_t st[3] = {b->stream, b->copy_stream, b->out_stream};
    float best = 0.f;
    for (int i = 0; i < 3; ++i) CU(cudaEventRecord(b->t1[i], st[i]));
    for (int i = 0; i < 3; ++i) {
        float ms = 0.f;
        CU(cudaEventSynchronize(b->t1[i]));
        CU(cudaEventElapsedTime(&ms, b->t0, b->t1[i]));
        best = ms > best ? ms : best;
    }
    *ms_out = best;
    return EKF_OK;
}
#if EKF_TILE_PROF
// development builds only: per-phase clock totals of the tile kernel since the last call (then reset)
int ekf_debug_tile_prof(uint64_t* out16) {
    unsigned long long v[16];
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(v, tile::g_tile_prof, sizeof(v)));
    for (int k = 0; k < 16; ++k) out16[k] = v[k];
    unsigned long long z[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    CU(cudaMemcpyToSymbol(tile::g_tile_prof, z, sizeof(z)));
    return EKF_OK;
}
#endif
int ekf_batch_launch_count(ekf_batch* b, uint64_t* out) {
    if (!b || !out) return fail(EKF_ERR_INVALID, "null argument");
    *out = b->launches;
    return EKF_OK;
}

int ekf_normalize_angles(const double* in, double* out, int64_t count, int device) {
    if (!in || !out || count < 0) return fail(EKF_ERR_INVALID, "invalid argument");
    if (count == 0) return EKF_OK;
    int rc = check_device(device);
    if (rc) return rc;
    DeviceGuard g(device);
    double *d_in = nullptr, *d_out = nullptr;
    CU(cudaMalloc(&d_in, sizeof(double) * count));
    CU(cudaMalloc(&d_out, sizeof(double) * count));
    CU(cudaMemcpy(d_in, in, sizeof(double) * count, cudaMemcpyHostToDevice));
    k_normalize<<<(unsigned)((count + 255) / 256), 256>>>(d_in, d_out, count);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, d_out, sizeof(double) * count, cudaMemcpyDeviceToHost));
    cudaFree(d_in);
    cudaFree(d_out);
    return EKF_OK;
}

// DiffDrive::updatePose for `count` independent odometers (rigid2d/src/diff_drive.cpp:50-67, integrateTwist
// rigid2d.cpp:304-333): poses [count][3] = {x, y, theta} in place, left / right wheel angle increments [count].
int ekf_update_pose(double wheel_base, double wheel_radius, int64_t count, double* poses, const double* left,
                    const double* right) {
    if (count < 0 || (count > 0 && (!poses || !left || !right))) return fail(EKF_ERR_INVALID, "invalid argument");
    if (count == 0) return EKF_OK;
    int ndev = 0;
    int rc = ekf_device_count(&ndev);
    if (rc) return rc;
    double *d_p = nullptr, *d_l = nullptr, *d_r = nullptr;
    cudaError_t e = cudaMalloc(&d_p, sizeof(double) * 3 * (size_t)count);
    if (e == cudaSuccess) e = cudaMalloc(&d_l, sizeof(double) * (size_t)count);
    if (e == cudaSuccess) e = cudaMalloc(&d_r, sizeof(double) * (size_t)count);
    if (e == cudaSuccess) e = cudaMemcpy(d_p, poses, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_l, left, sizeof(double) * (size_t)count, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_r, right, sizeof(double) * (size_t)count, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_update_pose<<<(unsigned)((count + 255) / 256), 256>>>(wheel_base, wheel_radius, count, d_p, d_l, d_r);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(poses, d_p, sizeof(double) * 3 * (size_t)count, cudaMemcpyDeviceToHost);
    cudaFree(d_p);
    cudaFree(d_l);
    cudaFree(d_r);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail((int)e, "ekf_update_pose: %s", cudaGetErrorString(e));
    }
    return EKF_OK;
}

// DiffDrive::getBodyTwistForUpdate, rigid2d/src/diff_drive.cpp:38-47 (two multiplies: host arithmetic)
int ekf_body_twist(double wheel_base, double wheel_radius, double left, double right, double* out2) {
    if (!out2) return fail(EKF_ERR_INVALID, "null argument");
    const double D = wheel_base * 0.5, r = wheel_radius;
    out2[0] = (r / (2.0 * D)) * (right - left);
    out2[1] = (r / 2.0) * (right + left);
    return EKF_OK;
}

}  // extern "C"
