// Host helpers of the C ABI sources (capi.cu, circles.cu, tubeworld.cu, sharded/sharded.cu).  Everything is in an
// anonymous namespace: each translation unit keeps its own error buffer, so every library's *_last_error() reports
// only its own errors.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <type_traits>

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            cudaGetLastError();                                                                          \
            return fail((int)e_, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                                \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// 0 when `device` is a visible CUDA device; otherwise the error (-1 for an index out of range).
int check_device(int device) {
    int count = 0;
    const cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail((int)e, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return fail(-1, "device %d not available (%d visible)", device, count);
    return 0;
}

// Launch with the programmatic-stream-serialization attribute (see pdl_prologue in ekf_large.cuh): only for kernels
// that start with pdl_prologue().
template <class... KArgs, class... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Runtime flags to compile-time ones: with_flags(f, b0, b1, ...) calls f(std::bool_constant<b0>{},
// std::bool_constant<b1>{}, ...), so that a generic lambda can instantiate the kernel variant the flags select.
template <class F>
decltype(auto) with_flags(F&& f) {
    return f();
}
template <class F, class... Flags>
decltype(auto) with_flags(F&& f, bool b, Flags... rest) {
    if (b) return with_flags([&](auto... c) { return f(std::true_type{}, c...); }, rest...);
    return with_flags([&](auto... c) { return f(std::false_type{}, c...); }, rest...);
}

// Set-up of one kernel on `device` (the current device), cached per kernel and device: raises the kernel's dynamic
// shared-memory limit to `smem` bytes when more is asked for than before (and then, with `max_carveout`, prefers the
// largest shared-memory carveout), and stores in *per_sm the CTAs of `threads` threads resident per SM at the size
// enabled.  Devices beyond the cache redo the set-up on every call.
template <auto Kernel>
cudaError_t kernel_setup(int device, int threads, int smem, bool max_carveout, int* per_sm = nullptr) {
    constexpr int kMaxDevices = 64;
    struct Entry {
        int smem = -1, per_sm = 0;
    };
    static Entry cache[kMaxDevices];
    Entry uncached;
    Entry& c = device >= 0 && device < kMaxDevices ? cache[device] : uncached;
    if (c.smem < smem) {
        cudaError_t e = cudaSuccess;
        if (smem > 0) e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess && smem > 0 && max_carveout)
            e = cudaFuncSetAttribute(Kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        int nb = 0;
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, Kernel, threads, smem);
        if (e != cudaSuccess) return e;
        c.smem = smem;
        c.per_sm = nb;
    }
    if (per_sm) *per_sm = c.per_sm;
    return cudaSuccess;
}

}  // namespace
