// cuda_owners.h -- move-only owners of the CUDA resources of the host code.  Each frees its resource in its destructor,
// so that every path out of a function, an error return included, leaves nothing behind.  Host only: the destructors
// do not switch devices, so an owner of another device's resource dies with that device current.
#ifndef GDX_CUDA_OWNERS_H
#define GDX_CUDA_OWNERS_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

namespace gdx {

// one device allocation: an image, an accelerator table, a temporary of a build, a grow-only buffer of a workspace
struct DevMem {
    void *p = nullptr;
    uint64_t bytes = 0;  // allocated
    DevMem() = default;
    DevMem(void *block, uint64_t nbytes) : p(block), bytes(nbytes) {}  // takes over a cudaMalloc'ed block
    DevMem(DevMem &&o) noexcept : p(std::exchange(o.p, nullptr)), bytes(std::exchange(o.bytes, 0)) {}
    DevMem &operator=(DevMem &&o) noexcept {
        std::swap(p, o.p);
        std::swap(bytes, o.bytes);
        return *this;
    }
    ~DevMem() { reset(); }
    void reset() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    // a block of nbytes (one byte for 0) in place of the old one, which is freed first; empty on failure
    cudaError_t alloc(uint64_t nbytes) {
        reset();
        const cudaError_t e = cudaMalloc(&p, nbytes ? nbytes : 1);
        if (e != cudaSuccess) p = nullptr;
        else bytes = nbytes;
        return e;
    }
    // grow-only: a block of at least nbytes.  The old block goes first; then 1/8 more than asked for, and the exact
    // size (rounded to 256 bytes) when that does not fit.
    cudaError_t reserve(uint64_t nbytes) {
        if (nbytes <= bytes) return cudaSuccess;
        const cudaError_t e = alloc((nbytes + nbytes / 8 + 255) / 256 * 256);
        return e == cudaSuccess ? e : alloc((nbytes + 255) / 256 * 256);
    }
    // the block to a new owner, which frees it
    void *release() {
        bytes = 0;
        return std::exchange(p, nullptr);
    }
    explicit operator bool() const { return p != nullptr; }
    template <class T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

// one pinned host allocation (staging for callers that pass ordinary pageable memory, words shared with kernels)
struct HBuf {
    void *p = nullptr;
    uint64_t bytes = 0;  // allocated
    HBuf() = default;
    HBuf(HBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), bytes(std::exchange(o.bytes, 0)) {}
    HBuf &operator=(HBuf &&o) noexcept {
        std::swap(p, o.p);
        std::swap(bytes, o.bytes);
        return *this;
    }
    ~HBuf() { reset(); }
    void reset() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
    }
    // exactly nbytes in place of the old block, which is freed first; empty on failure
    cudaError_t alloc(uint64_t nbytes) {
        reset();
        const cudaError_t e = cudaMallocHost(&p, nbytes);
        if (e != cudaSuccess) p = nullptr;
        else bytes = nbytes;
        return e;
    }
    // grow-only: the old block goes first, then 1/8 more than asked for, rounded to 4096 bytes
    cudaError_t reserve(uint64_t nbytes) {
        if (nbytes <= bytes) return cudaSuccess;
        return alloc((nbytes + nbytes / 8 + 4095) / 4096 * 4096);
    }
    template <class T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

// a block of the device's stream-ordered pool, freed on the stream it was allocated on
struct AsyncMem {
    void *p = nullptr;
    cudaStream_t stream = nullptr;
    AsyncMem() = default;
    AsyncMem(AsyncMem &&o) noexcept : p(std::exchange(o.p, nullptr)), stream(o.stream) {}
    AsyncMem &operator=(AsyncMem &&o) noexcept {
        std::swap(p, o.p);
        std::swap(stream, o.stream);
        return *this;
    }
    ~AsyncMem() { free(); }
    cudaError_t alloc(uint64_t nbytes, cudaStream_t st) {
        free();
        stream = st;
        const cudaError_t e = cudaMallocAsync(&p, nbytes, st);
        if (e != cudaSuccess) p = nullptr;
        return e;
    }
    // the block back to the pool, in stream order; the error of cudaFreeAsync
    cudaError_t free() { return p ? cudaFreeAsync(std::exchange(p, nullptr), stream) : cudaSuccess; }
    template <class T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

struct Event {
    cudaEvent_t ev = nullptr;
    Event() = default;
    Event(Event &&o) noexcept : ev(std::exchange(o.ev, nullptr)) {}
    Event &operator=(Event &&o) noexcept {
        std::swap(ev, o.ev);
        return *this;
    }
    ~Event() {
        if (ev) cudaEventDestroy(ev);
    }
    cudaError_t create(unsigned flags) {
        *this = Event();
        const cudaError_t e = cudaEventCreateWithFlags(&ev, flags);
        if (e != cudaSuccess) ev = nullptr;
        return e;
    }
    operator cudaEvent_t() const { return ev; }
};

struct Stream {
    cudaStream_t st = nullptr;
    Stream() = default;
    Stream(Stream &&o) noexcept : st(std::exchange(o.st, nullptr)) {}
    Stream &operator=(Stream &&o) noexcept {
        std::swap(st, o.st);
        return *this;
    }
    ~Stream() {
        if (st) cudaStreamDestroy(st);
    }
    cudaError_t create(unsigned flags) {
        *this = Stream();
        const cudaError_t e = cudaStreamCreateWithFlags(&st, flags);
        if (e != cudaSuccess) st = nullptr;
        return e;
    }
    operator cudaStream_t() const { return st; }
};

}  // namespace gdx
#endif
