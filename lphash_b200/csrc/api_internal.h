// Shared by the translation units behind the C ABI (c_api.cu, scan_api.cu, build_session.cu, build_api.cu): error
// slot, CUDA error propagation, the exception fence every entry point runs inside, owners of device resources, the
// layout of a batch of contigs.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
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
// a device allocation that failed for want of memory (a CudaError to every caller that does not ask for the size)
struct DeviceOom : CudaError {
    uint64_t bytes;
};

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
        const cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaErrorMemoryAllocation) {
            p = nullptr;
            throw DeviceOom{{e, "cudaMalloc(&p, want)"}, want};
        }
        CK(e);
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

// Layout of a batch of contigs (host offsets): max(0, L-k+1) k-mers per contig and, with m, max(0, L-m+1) m-mers.
// With code_offsets, writes where each contig's codes start (n_contigs + 1 entries).  Offsets that decrease are
// an argument error (thrown; guarded() reports it as LPHB_E_ARG).
struct ContigCounts {
    uint64_t kmers = 0, mmers = 0;
};
inline ContigCounts contig_layout(const uint64_t* offsets, uint64_t n_contigs, uint32_t k, uint32_t m = 0,
                                  uint64_t* code_offsets = nullptr) {
    ContigCounts n;
    for (uint64_t c = 0; c < n_contigs; ++c) {
        if (offsets[c + 1] < offsets[c]) throw std::invalid_argument("offsets must be non-decreasing");
        const uint64_t len = offsets[c + 1] - offsets[c];
        if (code_offsets) code_offsets[c] = n.kmers;
        n.kmers += len >= k ? len - k + 1 : 0;
        if (m) n.mmers += len >= m ? len - m + 1 : 0;
    }
    if (code_offsets) code_offsets[n_contigs] = n.kmers;
    return n;
}

// The (k, m) the build side takes (the scan and build sessions): the error text when (k, m) is outside, else null.
inline const char* scan_km_error(uint32_t k, uint32_t m) {
    return m == 0 || m > 31 || k < m || k > 63 ? "need 1 <= m <= 31, m <= k <= 63" : nullptr;
}

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
