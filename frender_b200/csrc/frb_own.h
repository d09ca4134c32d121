// Scoped owners of the CUDA resources of the host code (frb_lib.cu and the frb_*.inl files it includes): a buffer,
// event or stream is released when its owner goes out of scope, is reset or is assigned another, so a CU / TRY that
// returns early leaks nothing.  Move-only; nothing here throws.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>

namespace frb {

// Where a buffer comes from and goes back to.  `s` orders a pool allocation and its release; the other kinds ignore it.
struct DeviceMem {
    static cudaError_t acquire(void** p, size_t bytes, cudaStream_t) { return cudaMalloc(p, bytes); }
    static cudaError_t release(void* p, cudaStream_t) { return cudaFree(p); }
};
struct PinnedMem {
    static cudaError_t acquire(void** p, size_t bytes, cudaStream_t) { return cudaMallocHost(p, bytes); }
    static cudaError_t release(void* p, cudaStream_t) { return cudaFreeHost(p); }
};
// Stream-ordered, from the device's memory pool (whose release threshold frb_create sets to "never", so a steady-state
// step makes no driver call that synchronises the device).  An empty request still takes 8 bytes.
struct PoolMem {
    static cudaError_t acquire(void** p, size_t bytes, cudaStream_t s) { return cudaMallocAsync(p, bytes ? bytes : 8, s); }
    static cudaError_t release(void* p, cudaStream_t s) { return cudaFreeAsync(p, s); }
};

// n elements of T.  It converts to T*, so it goes wherever the pointer went.
template <typename T, typename Kind>
class Buf {
  public:
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    Buf(Buf&& o) noexcept : p_(o.p_), n_(o.n_), s_(o.s_) { o.p_ = nullptr, o.n_ = 0; }
    Buf& operator=(Buf&& o) noexcept {
        if (this != &o) {
            reset();
            p_ = o.p_, n_ = o.n_, s_ = o.s_;
            o.p_ = nullptr, o.n_ = 0;
        }
        return *this;
    }
    ~Buf() { reset(); }

    // n elements in place of what the buffer held, which is released first (the two never coexist).  On failure the
    // buffer is empty and the runtime's last error is cleared, so that no later cudaGetLastError reports it again.
    cudaError_t alloc(size_t n, cudaStream_t s = nullptr) {
        reset();
        void* p = nullptr;
        const cudaError_t e = Kind::acquire(&p, n * sizeof(T), s);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return e;
        }
        p_ = static_cast<T*>(p), n_ = n, s_ = s;
        return cudaSuccess;
    }
    void reset() {
        if (p_) Kind::release(p_, s_);
        p_ = nullptr, n_ = 0;
    }
    T* get() const { return p_; }
    operator T*() const { return p_; }
    T* operator->() const { return p_; }
    size_t size() const { return n_; }

  private:
    T* p_ = nullptr;
    size_t n_ = 0;
    cudaStream_t s_ = nullptr;
};

template <typename T>
using DevBuf = Buf<T, DeviceMem>;
template <typename T>
using PinnedBuf = Buf<T, PinnedMem>;
template <typename T>
using PoolBuf = Buf<T, PoolMem>;  // alloc(n, stream)

// An event or a stream, created with flags.
template <typename H, cudaError_t (*Create)(H*, unsigned), cudaError_t (*Destroy)(H)>
class Handle {
  public:
    Handle() = default;
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;
    Handle(Handle&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    Handle& operator=(Handle&& o) noexcept {
        if (this != &o) {
            reset();
            h_ = o.h_;
            o.h_ = nullptr;
        }
        return *this;
    }
    ~Handle() { reset(); }

    cudaError_t create(unsigned flags) {
        reset();
        const cudaError_t e = Create(&h_, flags);
        if (e != cudaSuccess) {
            h_ = nullptr;
            cudaGetLastError();
        }
        return e;
    }
    void reset() {
        if (h_) Destroy(h_);
        h_ = nullptr;
    }
    operator H() const { return h_; }

  private:
    H h_ = nullptr;
};

using Event = Handle<cudaEvent_t, cudaEventCreateWithFlags, cudaEventDestroy>;
using Stream = Handle<cudaStream_t, cudaStreamCreateWithFlags, cudaStreamDestroy>;

}  // namespace frb
