// Owners of the library's device memory: one cudaMalloc allocation (DevBuf) and one CUDA IPC mapping of a peer's
// allocation (IpcMapping).  Both are move-only and give back what they hold in their destructors; this header is the
// only place that frees device memory or closes a mapping.  copy_to_device is how host data reaches that memory.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstddef>
#include <cstdint>
#include <utility>

namespace kr {

// allocations and mappings currently owned by a DevBuf or an IpcMapping, process-wide (krotov_live_device_objects)
inline std::atomic<int64_t> g_live_device_objects{0};

class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p_(std::exchange(o.p_, nullptr)), bytes_(std::exchange(o.bytes_, 0)) {}
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) {
            reset();
            p_ = std::exchange(o.p_, nullptr);
            bytes_ = std::exchange(o.bytes_, 0);
        }
        return *this;
    }
    ~DevBuf() { reset(); }

    // frees the current allocation, then allocates `bytes`; the buffer is empty when the allocation fails
    cudaError_t allocate(size_t bytes) {
        reset();
        void *p = nullptr;
        const cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return e;
        p_ = p;
        bytes_ = bytes;
        ++g_live_device_objects;
        return cudaSuccess;
    }
    void reset() {
        if (p_) {
            cudaFree(p_);
            --g_live_device_objects;
        }
        p_ = nullptr;
        bytes_ = 0;
    }
    size_t bytes() const { return bytes_; }
    template <typename T>
    T *get() const {
        return static_cast<T *>(p_);
    }
    explicit operator bool() const { return p_ != nullptr; }

  private:
    void *p_ = nullptr;
    size_t bytes_ = 0;
};

class IpcMapping {
  public:
    IpcMapping() = default;
    IpcMapping(const IpcMapping &) = delete;
    IpcMapping &operator=(const IpcMapping &) = delete;
    IpcMapping(IpcMapping &&o) noexcept : p_(std::exchange(o.p_, nullptr)) {}
    IpcMapping &operator=(IpcMapping &&o) noexcept {
        if (this != &o) {
            reset();
            p_ = std::exchange(o.p_, nullptr);
        }
        return *this;
    }
    ~IpcMapping() { reset(); }

    // closes the current mapping, then maps the peer allocation `mh`; the mapping is empty when that fails
    cudaError_t open(const cudaIpcMemHandle_t &mh) {
        reset();
        void *p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return e;
        p_ = p;
        ++g_live_device_objects;
        return cudaSuccess;
    }
    void reset() {
        if (p_) {
            cudaIpcCloseMemHandle(p_);
            --g_live_device_objects;
        }
        p_ = nullptr;
    }
    template <typename T>
    T *get() const {
        return static_cast<T *>(p_);
    }

  private:
    void *p_ = nullptr;
};

// Copies `bytes` from host memory to device memory on `stream`, the stream of the handle that owns `dst`.  Every write
// to the library's device memory is ordered on that stream: the sweeps run there, it is non-blocking, so nothing orders
// it after work on the legacy stream, and a blocking cudaMemcpy from pageable memory may return before its DMA lands.
// The copy may read `src` after this returns: `wait` waits for it, so that the caller may then free or rewrite `src`.
inline cudaError_t copy_to_device(void *dst, const void *src, size_t bytes, cudaStream_t stream, bool wait) {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess && wait) e = cudaStreamSynchronize(stream);
    return e;
}

}  // namespace kr
