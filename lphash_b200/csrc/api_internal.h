// Shared by the translation units behind the C ABI (c_api.cu, build_api.cu): error slot, CUDA error
// propagation, the exception fence every entry point runs inside, owners of device resources.
#pragma once
#include <cuda_runtime.h>

#include <new>
#include <stdexcept>
#include <string>
#include <utility>

#include "../../include/lphash_b200.h"
#include "lph_image.h"

namespace lphb {

std::string& last_error_slot();  // thread-local; read by lphb_last_error (c_api.cu)

inline int fail(int code, std::string const& msg) {
    last_error_slot() = msg;
    return code;
}

struct CudaError {
    cudaError_t e;
    const char* what;
};
#define CK(expr)                                              \
    do {                                                      \
        cudaError_t e__ = (expr);                             \
        if (e__ != cudaSuccess) throw ::lphb::CudaError{e__, #expr}; \
    } while (0)

// The owners below free what they hold when they go out of scope, ignoring errors; the device that owns the
// resource must be current then.

// grow-only device buffer
struct DevBuf {
    void* p = nullptr;
    uint64_t cap = 0;
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    void reserve(uint64_t bytes) {
        if (bytes <= cap) return;
        if (p) CK(cudaFree(p));
        p = nullptr;
        cap = 0;
        uint64_t want = bytes + bytes / 8 + 256;
        CK(cudaMalloc(&p, want));
        cap = want;
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

// grow-only pinned host buffer
struct HostBuf {
    void* p = nullptr;
    uint64_t cap = 0;
    HostBuf() = default;
    HostBuf(HostBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    ~HostBuf() {
        if (p) cudaFreeHost(p);
    }
    void reserve(uint64_t bytes) {
        if (bytes <= cap) return;
        if (p) CK(cudaFreeHost(p));
        p = nullptr;
        cap = 0;
        CK(cudaMallocHost(&p, bytes));
        cap = bytes;
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

// non-blocking stream, created on first use
struct Stream {
    cudaStream_t s = nullptr;
    Stream() = default;
    Stream(Stream&& o) noexcept : s(std::exchange(o.s, nullptr)) {}
    ~Stream() {
        if (s) cudaStreamDestroy(s);
    }
    void create() {
        if (!s) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    }
    operator cudaStream_t() const { return s; }
};

struct Event {
    cudaEvent_t e = nullptr;
    Event() = default;
    Event(Event&& o) noexcept : e(std::exchange(o.e, nullptr)) {}
    ~Event() {
        if (e) cudaEventDestroy(e);
    }
    void create(unsigned flags) {
        if (!e) CK(cudaEventCreateWithFlags(&e, flags));
    }
    operator cudaEvent_t() const { return e; }
};

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        CK(cudaGetDevice(&prev));
        if (prev != dev) CK(cudaSetDevice(dev));
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// nothing may cross the C boundary as an exception
template <class F>
int guarded(F&& body) {
    try {
        return body();
    } catch (CudaError const& e) {
        cudaGetLastError();
        return fail(LPHB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e.e) + " in " + e.what);
    } catch (FormatError const& e) {
        return fail(LPHB_E_FORMAT, e.what());
    } catch (std::bad_alloc const&) {
        return fail(LPHB_E_NOMEM, "out of host memory");
    } catch (std::exception const& e) {
        return fail(LPHB_E_ARG, e.what());
    }
}

}  // namespace lphb
