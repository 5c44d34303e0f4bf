// hlynr_host.cuh -- host-side helpers shared by the translation units of the library (internal: not part of include/ or the ABI).
#pragma once

#include <memory>
#include <type_traits>

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

// Owners of the CUDA resources a handle allocates: each releases what it holds when it is destroyed or re-assigned, so a
// handle's destructor frees everything and an allocation repeated after a failure leaks nothing.  The resources belong to the
// device that was current when they were made; the owner must be destroyed with that device current (a DeviceGuard).
struct CudaFree { void operator()(void* p) const { cudaFree(p); } };
struct CudaFreeHost { void operator()(void* p) const { cudaFreeHost(p); } };
struct CudaStreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct CudaEventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
template <class T> using DevPtr = std::unique_ptr<T, CudaFree>;       // device memory
template <class T> using PinnedPtr = std::unique_ptr<T, CudaFreeHost>;  // page-locked host memory
using StreamOwner = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, CudaStreamDestroy>;
using EventOwner = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, CudaEventDestroy>;

// The helpers below replace what the owner held, and leave it empty if the call fails; use them under CK.
// `count` elements of device memory (DevPtr) or page-locked host memory (PinnedPtr); the old block is freed first.
template <class T, class D> cudaError_t alloc(std::unique_ptr<T, D>& p, size_t count) {
    static_assert(std::is_same<D, CudaFree>::value || std::is_same<D, CudaFreeHost>::value, "a DevPtr or a PinnedPtr");
    p.reset();
    void* q = nullptr;
    const cudaError_t e = std::is_same<D, CudaFree>::value ? cudaMalloc(&q, count * sizeof(T)) : cudaMallocHost(&q, count * sizeof(T));
    if (e == cudaSuccess) p.reset(static_cast<T*>(q));
    return e;
}
// a stream that does not synchronise with the legacy default stream
inline cudaError_t stream_create(StreamOwner& s) {
    cudaStream_t q = nullptr;
    const cudaError_t e = cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking);
    s.reset(e == cudaSuccess ? q : nullptr);
    return e;
}
// an event for ordering only (no timing)
inline cudaError_t event_create(EventOwner& ev) {
    cudaEvent_t q = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&q, cudaEventDisableTiming);
    ev.reset(e == cudaSuccess ? q : nullptr);
    return e;
}
