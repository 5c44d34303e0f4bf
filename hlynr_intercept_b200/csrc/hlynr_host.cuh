// hlynr_host.cuh -- host-side helpers shared by the translation units of the library (internal: not part of include/ or the ABI).
#pragma once

#include <cuda_runtime.h>

// Formats the message into the calling thread's hlynr_last_error() and returns 1 (defined in hlynr_capi.cu).
extern "C" int hlynr_internal_fail(const char* fmt, ...);
inline constexpr int (&fail)(const char*, ...) = hlynr_internal_fail;

// Returns fail(...) from the enclosing function if a CUDA runtime call does not succeed.
#define CK(call)                                                                                                                   \
    do {                                                                                                                           \
        cudaError_t _e = (call);                                                                                                   \
        if (_e != cudaSuccess) return fail("%s: %s failed: %s (%s:%d)", __func__, #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

// Fails (`who` names the entry point) if `st` is capturing a CUDA graph: for the calls that must not be recorded into one.
inline int refuse_capture(cudaStream_t st, const char* who) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    const cudaError_t e = cudaStreamIsCapturing(st, &cs);
    if (e != cudaSuccess) return fail("%s: cudaStreamIsCapturing failed: %s", who, cudaGetErrorString(e));
    if (cs != cudaStreamCaptureStatusNone) return fail("%s: refused while the stream is capturing a CUDA graph", who);
    return 0;
}

// Makes `dev` the current device for the scope and restores the caller's device on exit; ok is false if it could not be selected.
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
