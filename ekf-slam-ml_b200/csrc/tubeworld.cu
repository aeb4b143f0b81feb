// Batched on-device input generator (include/tube_world_b200.h): the simulator side of the reference
// (nurtlesim/src/tube_world.cpp) for B independent robots, one thread per robot (per robot and beam for the laser).
// Arithmetic mirrors ekf-slam-ml_b200/tracegen.py operation for operation; the hash RNG is integer-exact, the
// transcendental functions differ from numpy's in the last bits only.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <new>

#include "../../include/tube_world_b200.h"
#include "ekf_math.cuh"
#include "host_util.cuh"

namespace tw {

using ekf::kPi;
using ekf::kTwoPi;

constexpr unsigned long long M1 = 0x9E3779B97F4A7C15ull, M2 = 0xBF58476D1CE4E5B9ull, M3 = 0x94D049BB133111EBull;

__device__ __forceinline__ unsigned long long mix(unsigned long long z) {
    z ^= z >> 30;
    z *= M2;
    z ^= z >> 27;
    z *= M3;
    z ^= z >> 31;
    return z;
}
// U(0,1), never 0: tracegen.hash_uniform
__device__ __forceinline__ double hash_uniform(unsigned long long seed, unsigned long long filt, unsigned long long ctr) {
    unsigned long long z = seed * M1 + filt * M2 + ctr * M3 + 0x1234567ull;
    z = mix(mix(z) + M1);
    return ((double)(z >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}
// N(0,1) by Box-Muller: tracegen.hash_normal
__device__ __forceinline__ double hash_normal(unsigned long long seed, unsigned long long filt, unsigned long long ctr) {
    const double u1 = hash_uniform(seed, filt, ctr);
    const double u2 = hash_uniform(seed, filt, ctr + (1ull << 40));
    return sqrt(-2.0 * log(u1)) * cos(kTwoPi * u2);
}
__device__ __forceinline__ unsigned long long ctr_of(long long tick, int purpose, int sub) {
    return (unsigned long long)tick * 4096ull + (unsigned long long)(purpose * 512 + sub);
}

struct Robots {
    double *x, *y, *th, *v, *om, *dl, *dr;
    double *ox, *oy, *oth;  // dead-reckoning odometer (slam.cpp:96): same wheel increments, no collisions
};

// one simulator tick of one robot (tube_world.cpp:193-250, 316-366), tracegen.TubeWorldSim.step_tick
__device__ __forceinline__ void tick_once(const tubeworld_params& p, const double* __restrict__ tx,
                                          const double* __restrict__ ty, int n_tubes, unsigned long long seed,
                                          unsigned long long fid, long long tick, double& x, double& y, double& th,
                                          double& v, double& om, double& dl, double& dr, double& ox, double& oy,
                                          double& oth) {
    if (tick % 10 == 0) {
        v = p.cmd_v + p.vx_std * hash_normal(seed, fid, ctr_of(tick, 0, 0));
        om = p.cmd_v / p.cmd_radius + p.the_std * hash_normal(seed, fid, ctr_of(tick, 1, 0));
    }
    const double D = p.wheel_base * 0.5, r = p.wheel_radius;
    const double wl = -(D / r) * om + (1.0 / r) * v;
    const double wr = (D / r) * om + (1.0 / r) * v;
    const double span = p.slip_max - p.slip_min;
    dl = (wl / 100.0) * (p.slip_min + span * hash_uniform(seed, fid, ctr_of(tick, 2, 0)));
    dr = (wr / 100.0) * (p.slip_min + span * hash_uniform(seed, fid, ctr_of(tick, 3, 0)));
    const double om_b = (r / (2.0 * D)) * (dr - dl);
    const double vx_b = (r / 2.0) * (dr + dl);
    const bool turning = fabs(om_b) > 0.0001;
    double bx = vx_b, by = 0.0, dth = 0.0;
    if (turning) {
        double so, co;
        sincos(om_b, &so, &co);
        bx = (vx_b / om_b) * so;
        by = (vx_b / om_b) * (1.0 - co);
        dth = om_b;
    }
    double s, c;
    sincos(th, &s, &c);
    x = x + c * bx - s * by;
    y = y + s * bx + c * by;
    th = th + dth;
    double so_, co_;
    sincos(oth, &so_, &co_);
    ox = ox + co_ * bx - so_ * by;
    oy = oy + so_ * bx + co_ * by;
    oth = oth + dth;
    const double lim = p.tube_radius + p.wheel_base / 2;
    for (int j = 0; j < n_tubes; ++j) {  // first tube closer than the limit snaps the robot back
        const double dx = tx[j] - x, dy = ty[j] - y;
        if (hypot(dx, dy) < lim) {
            const double ang = atan2(dy, dx);
            double sa, ca;
            sincos(ang, &sa, &ca);
            x = tx[j] - lim * ca;
            y = ty[j] - lim * sa;
            break;
        }
    }
}

__global__ void __launch_bounds__(128)
    k_step_known(tubeworld_params p, const double* __restrict__ tx, const double* __restrict__ ty, int n_tubes,
                 unsigned long long seed, long long first_filter, long long B, long long tick0, int n_ticks, Robots R,
                 int report_visible, double* __restrict__ twists, double* __restrict__ xy, uint8_t* __restrict__ vis,
                 double* __restrict__ truth, double* __restrict__ odom) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const unsigned long long fid = (unsigned long long)(first_filter + b);
    double x = R.x[b], y = R.y[b], th = R.th[b], v = R.v[b], om = R.om[b], dl = R.dl[b], dr = R.dr[b];
    double ox = R.ox[b], oy = R.oy[b], oth = R.oth[b];
    for (int k = 0; k < n_ticks; ++k)
        tick_once(p, tx, ty, n_tubes, seed, fid, tick0 + k, x, y, th, v, om, dl, dr, ox, oy, oth);
    R.x[b] = x, R.y[b] = y, R.th[b] = th, R.v[b] = v, R.om[b] = om, R.dl[b] = dl, R.dr[b] = dr;
    R.ox[b] = ox, R.oy[b] = oy, R.oth[b] = oth;
    odom[3 * b] = ox, odom[3 * b + 1] = oy, odom[3 * b + 2] = oth;
    const long long tick = tick0 + n_ticks;
    // odometry twist handed to prediction(): getBodyTwistForUpdate(10 dl, 10 dr)  (slam.cpp:173-176)
    const double D = p.wheel_base * 0.5, r = p.wheel_radius;
    const double l10 = dl * 10.0, r10 = dr * 10.0;
    twists[2 * b] = (r / (2.0 * D)) * (r10 - l10);
    twists[2 * b + 1] = (r / 2.0) * (r10 + l10);
    truth[3 * b] = x, truth[3 * b + 1] = y, truth[3 * b + 2] = th;
    // fake sensor (tube_world.cpp:369-414)
    double s, c;
    sincos(th, &s, &c);
    const int n = p.n_slots, nt = n_tubes < n ? n_tubes : n;
    for (int j = 0; j < nt; ++j) {
        const double dx = tx[j] - x, dy = ty[j] - y;
        const double rx = c * dx + s * dy, ry = -s * dx + c * dy;
        const double nx = hash_normal(seed, fid, ctr_of(tick, 4, 2 * j));
        const double ny = hash_normal(seed, fid, ctr_of(tick, 4, 2 * j + 1));
        xy[b * 2 * n + 2 * j] = rx + p.sensor_std * nx;
        xy[b * 2 * n + 2 * j + 1] = ry + p.sensor_std * ny;
        vis[b * n + j] = (report_visible && hypot(dx, dy) <= p.max_visible) ? 1 : 0;
    }
    for (int j = nt; j < n; ++j) {
        xy[b * 2 * n + 2 * j] = 0.0;
        xy[b * 2 * n + 2 * j + 1] = 0.0;
        vis[b * n + j] = 0;
    }
}

__global__ void __launch_bounds__(128)
    k_advance(tubeworld_params p, const double* __restrict__ tx, const double* __restrict__ ty, int n_tubes,
              unsigned long long seed, long long first_filter, long long B, long long tick0, int n_ticks, Robots R,
              double* __restrict__ twists, double* __restrict__ truth, double* __restrict__ odom) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const unsigned long long fid = (unsigned long long)(first_filter + b);
    double x = R.x[b], y = R.y[b], th = R.th[b], v = R.v[b], om = R.om[b], dl = R.dl[b], dr = R.dr[b];
    double ox = R.ox[b], oy = R.oy[b], oth = R.oth[b];
    for (int k = 0; k < n_ticks; ++k)
        tick_once(p, tx, ty, n_tubes, seed, fid, tick0 + k, x, y, th, v, om, dl, dr, ox, oy, oth);
    R.x[b] = x, R.y[b] = y, R.th[b] = th, R.v[b] = v, R.om[b] = om, R.dl[b] = dl, R.dr[b] = dr;
    R.ox[b] = ox, R.oy[b] = oy, R.oth[b] = oth;
    odom[3 * b] = ox, odom[3 * b + 1] = oy, odom[3 * b + 2] = oth;
    const double D = p.wheel_base * 0.5, r = p.wheel_radius;
    const double l10 = dl * 10.0, r10 = dr * 10.0;
    twists[2 * b] = (r / (2.0 * D)) * (r10 - l10);
    twists[2 * b + 1] = (r / 2.0) * (r10 + l10);
    truth[3 * b] = x, truth[3 * b + 1] = y, truth[3 * b + 2] = th;
}

// 360-beam ray cast with box walls and tubes (tube_world.cpp:423-577), tracegen.TubeWorldSim.laser_scan
__global__ void __launch_bounds__(128)
    k_scan(tubeworld_params p, const double* __restrict__ tx, const double* __restrict__ ty, int n_tubes,
           unsigned long long seed, long long first_filter, long long B, long long tick, int n_beams, Robots R,
           float* __restrict__ ranges) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= B * n_beams) return;
    const long long b = g / n_beams;
    const int i = (int)(g - b * n_beams);
    const unsigned long long fid = (unsigned long long)(first_filter + b);
    const double x = R.x[b], y = R.y[b], th = R.th[b];
    const double res = kTwoPi / (double)n_beams;
    const double curr = ekf::normalize_angle(res * (double)i);
    const double x_dis = p.border / 2.0 - x, y_dis = p.border / 2.0 - y;
    const double box_ang = ekf::normalize_angle(res * (double)i + th);
    const double y_t = box_ang < 0 ? -(p.border - y_dis) : y_dis;
    const double x_t = (box_ang > kPi / 2.0 || box_ang < -kPi / 2.0) ? -(p.border - x_dis) : x_dis;
    double sb, cb;
    sincos(box_ang, &sb, &cb);
    double min_r = fmin(fmin(x_t / cb, y_t / sb), 3.5);
    double s, c;
    sincos(th, &s, &c);
    double sc, cc;
    sincos(curr, &sc, &cc);
    const double half = atan2(p.tube_radius, 0.12);
    for (int m = 0; m < n_tubes; ++m) {
        const double dx = tx[m] - x, dy = ty[m] - y;
        const double tbx = c * dx + s * dy, tby = -s * dx + c * dy;  // tube in the robot frame
        const double bearing = atan2(tby, tbx);
        const double sbg = ekf::normalize_angle(bearing - half), ebg = ekf::normalize_angle(bearing + half);
        const bool inside = (curr > sbg) && (curr < ebg);
        const bool wrap = (sbg > 0) && (ebg < 0);
        const bool flag = wrap ? ((curr > sbg) || (curr < ebg)) : inside;
        if (!flag) continue;
        // getLineCircleIntersection in the tube frame
        const double x1 = -tbx, y1 = -tby;
        const double x2 = 3.5 * cc + x1, y2 = 3.5 * sc + y1;
        const double ddx = x2 - x1, ddy = y2 - y1;
        const double dr2 = ddx * ddx + ddy * ddy;
        const double Dd = x1 * y2 - x2 * y1;
        const double delta = p.tube_radius * p.tube_radius * dr2 - Dd * Dd;
        if (!(delta > 0)) continue;
        const double sq = sqrt(delta);
        const double sgn = ddy < 0 ? -1.0 : 1.0;
        const double ix1 = (Dd * ddy + sgn * ddx * sq) / dr2, iy1 = (-Dd * ddx + fabs(ddy) * sq) / dr2;
        const double ix2 = (Dd * ddy - sgn * ddx * sq) / dr2, iy2 = (-Dd * ddx - fabs(ddy) * sq) / dr2;
        const double d1 = hypot(x1 - ix1, y1 - iy1), d2 = hypot(x1 - ix2, y1 - iy2);
        min_r = fmin(min_r, fmin(d1, d2));
    }
    const double noise = hash_normal(seed, fid, ctr_of(tick, 6, i));
    ranges[g] = (float)(min_r + p.range_std * noise);
}

}  // namespace tw

struct tubeworld {
    long long B = 0, first_filter = 0, tick = 0;
    int n_tubes = 0, device = 0, n_beams_cap = 0, n_beams_last = 0, calls = 0;
    bool own_stream = true;
    unsigned long long seed = 0;
    tubeworld_params p{};
    cudaStream_t stream = nullptr;
    double *d_tx = nullptr, *d_ty = nullptr;
    double* d_robots = nullptr;  // 10 arrays of B
    tw::Robots R{};
    double *d_twists = nullptr, *d_xy = nullptr, *d_truth = nullptr, *d_odom = nullptr;
    uint8_t* d_vis = nullptr;
    float* d_ranges = nullptr;
};

extern "C" {

const char* tubeworld_last_error(void) { return g_err; }

int tubeworld_destroy(tubeworld* w) {
    if (!w) return 0;
    DeviceGuard g(w->device);
    /* a borrowed stream may already be gone when the consumer was closed first: never touch it here */
    if (w->stream && w->own_stream) cudaStreamSynchronize(w->stream);
    else cudaDeviceSynchronize();
    cudaFree(w->d_tx);
    cudaFree(w->d_ty);
    cudaFree(w->d_robots);
    cudaFree(w->d_twists);
    cudaFree(w->d_xy);
    cudaFree(w->d_truth);
    cudaFree(w->d_odom);
    cudaFree(w->d_vis);
    cudaFree(w->d_ranges);
    if (w->stream && w->own_stream) cudaStreamDestroy(w->stream);
    cudaGetLastError();
    delete w;
    return 0;
}

int tubeworld_create(int64_t B, const tubeworld_params* p, const double* tubes_x, const double* tubes_y, int n_tubes,
                     uint64_t seed, int64_t first_filter, int device, tubeworld** out) {
    if (!out) return fail(-1, "null out pointer");
    *out = nullptr;
    if (B <= 0 || !p || n_tubes < 0 || (n_tubes > 0 && (!tubes_x || !tubes_y)) || p->n_slots <= 0)
        return fail(-1, "invalid argument");
    if (n_tubes > 255) return fail(-2, "at most 255 tubes (RNG counter layout)");
    const int rc = check_device(device);
    if (rc) return rc;
    DeviceGuard g(device);
    tubeworld* w = new (std::nothrow) tubeworld();
    if (!w) return fail(-3, "out of host memory");
    w->B = B;
    w->first_filter = first_filter;
    w->seed = seed;
    w->n_tubes = n_tubes;
    w->device = device;
    w->p = *p;
    cudaError_t err = cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking);
    auto A = [&](void** ptr, size_t bytes) {
        if (err == cudaSuccess) err = cudaMalloc(ptr, bytes ? bytes : 8);
    };
    A((void**)&w->d_tx, sizeof(double) * n_tubes);
    A((void**)&w->d_ty, sizeof(double) * n_tubes);
    A((void**)&w->d_robots, sizeof(double) * 10 * (size_t)B);
    A((void**)&w->d_twists, sizeof(double) * 2 * (size_t)B);
    A((void**)&w->d_xy, sizeof(double) * 2 * (size_t)p->n_slots * (size_t)B);
    A((void**)&w->d_truth, sizeof(double) * 3 * (size_t)B);
    A((void**)&w->d_odom, sizeof(double) * 3 * (size_t)B);
    A((void**)&w->d_vis, (size_t)p->n_slots * (size_t)B);
    if (err == cudaSuccess && n_tubes) err = cudaMemcpyAsync(w->d_tx, tubes_x, sizeof(double) * n_tubes, cudaMemcpyHostToDevice, w->stream);
    if (err == cudaSuccess && n_tubes) err = cudaMemcpyAsync(w->d_ty, tubes_y, sizeof(double) * n_tubes, cudaMemcpyHostToDevice, w->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(w->d_robots, 0, sizeof(double) * 10 * (size_t)B, w->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(w->stream);
    if (err != cudaSuccess) {
        cudaGetLastError();
        int code = fail((int)err, "tubeworld_create: %s", cudaGetErrorString(err));
        tubeworld_destroy(w);
        return code;
    }
    double* r = w->d_robots;
    w->R = tw::Robots{r, r + B, r + 2 * B, r + 3 * B, r + 4 * B, r + 5 * B, r + 6 * B, r + 7 * B, r + 8 * B, r + 9 * B};
    *out = w;
    return 0;
}

int tubeworld_step_known(tubeworld* w) {
    if (!w) return fail(-1, "null handle");
    DeviceGuard g(w->device);
    const unsigned blocks = (unsigned)((w->B + 127) / 128);
    tw::k_step_known<<<blocks, 128, 0, w->stream>>>(w->p, w->d_tx, w->d_ty, w->n_tubes, w->seed, w->first_filter, w->B, w->tick,
                                                   11, w->R, w->calls > 0 ? 1 : 0, w->d_twists, w->d_xy, w->d_vis, w->d_truth,
                                                   w->d_odom);
    CU(cudaGetLastError());
    w->tick += 11;
    w->calls += 1;
    return 0;
}

int tubeworld_step_scan(tubeworld* w, int ticks, int n_beams) {
    if (!w || ticks < 0 || n_beams < 2 || n_beams > 511) return fail(-1, "invalid argument");
    DeviceGuard g(w->device);
    if (n_beams > w->n_beams_cap) {
        CU(cudaStreamSynchronize(w->stream));
        cudaFree(w->d_ranges);
        w->d_ranges = nullptr;
        CU(cudaMalloc((void**)&w->d_ranges, sizeof(float) * (size_t)n_beams * (size_t)w->B));
        w->n_beams_cap = n_beams;
    }
    if (ticks > 0) {
        tw::k_advance<<<(unsigned)((w->B + 127) / 128), 128, 0, w->stream>>>(w->p, w->d_tx, w->d_ty, w->n_tubes, w->seed,
                                                                            w->first_filter, w->B, w->tick, ticks, w->R,
                                                                            w->d_twists, w->d_truth, w->d_odom);
        w->tick += ticks;
    }
    const long long total = w->B * n_beams;
    tw::k_scan<<<(unsigned)((total + 127) / 128), 128, 0, w->stream>>>(w->p, w->d_tx, w->d_ty, w->n_tubes, w->seed,
                                                                     w->first_filter, w->B, w->tick, n_beams, w->R, w->d_ranges);
    CU(cudaGetLastError());
    w->n_beams_last = n_beams;
    return 0;
}

int tubeworld_outputs(tubeworld* w, void** d_twists, void** d_xy, void** d_vis, void** d_truth, void** d_ranges) {
    if (!w) return fail(-1, "null handle");
    if (d_twists) *d_twists = w->d_twists;
    if (d_xy) *d_xy = w->d_xy;
    if (d_vis) *d_vis = w->d_vis;
    if (d_truth) *d_truth = w->d_truth;
    if (d_ranges) *d_ranges = w->d_ranges;
    return 0;
}

int tubeworld_download(tubeworld* w, double* twists, double* xy, uint8_t* vis, double* truth, float* ranges) {
    if (!w) return fail(-1, "null handle");
    DeviceGuard g(w->device);
    const size_t B = (size_t)w->B, n = (size_t)w->p.n_slots;
    if (twists) CU(cudaMemcpyAsync(twists, w->d_twists, sizeof(double) * 2 * B, cudaMemcpyDeviceToHost, w->stream));
    if (xy) CU(cudaMemcpyAsync(xy, w->d_xy, sizeof(double) * 2 * n * B, cudaMemcpyDeviceToHost, w->stream));
    if (vis) CU(cudaMemcpyAsync(vis, w->d_vis, n * B, cudaMemcpyDeviceToHost, w->stream));
    if (truth) CU(cudaMemcpyAsync(truth, w->d_truth, sizeof(double) * 3 * B, cudaMemcpyDeviceToHost, w->stream));
    if (ranges) {
        if (!w->d_ranges) return fail(-3, "no scan has been generated yet");
        CU(cudaMemcpyAsync(ranges, w->d_ranges, sizeof(float) * (size_t)w->n_beams_last * B, cudaMemcpyDeviceToHost, w->stream));
    }
    CU(cudaStreamSynchronize(w->stream));
    return 0;
}

int tubeworld_odometry(tubeworld* w, void** d_odom, double* odom) {
    if (!w) return fail(-1, "null handle");
    if (d_odom) *d_odom = w->d_odom;
    if (odom) {
        DeviceGuard g(w->device);
        CU(cudaMemcpyAsync(odom, w->d_odom, sizeof(double) * 3 * (size_t)w->B, cudaMemcpyDeviceToHost, w->stream));
        CU(cudaStreamSynchronize(w->stream));
    }
    return 0;
}

int tubeworld_sync(tubeworld* w) {
    if (!w) return fail(-1, "null handle");
    DeviceGuard g(w->device);
    CU(cudaStreamSynchronize(w->stream));
    return 0;
}
void* tubeworld_stream(tubeworld* w) { return w ? (void*)w->stream : nullptr; }
// Run the generator on the consumer's stream (e.g. ekf_batch_stream()): generation and filtering are then
// stream-ordered and need no host synchronisation in between.
int tubeworld_set_stream(tubeworld* w, void* stream) {
    if (!w || !stream) return fail(-1, "null argument");
    DeviceGuard g(w->device);
    CU(cudaStreamSynchronize(w->stream));
    if (w->own_stream) cudaStreamDestroy(w->stream);
    w->stream = (cudaStream_t)stream;
    w->own_stream = false;
    return 0;
}

}  // extern "C"
