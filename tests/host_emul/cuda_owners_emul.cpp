// Host build of the CUDA owners (genedex_b200/csrc/cuda_owners.h) for tests/test_cuda_owners_host.py.  The runtime
// functions the owners call are defined here: they hand out malloc'ed blocks and counted handles, keep every live
// resource per kind, log the sizes asked for, and fail on request (the k-th acquiring call, or any allocation larger
// than a limit).  Freeing something that is not live is counted as a bad free.
#include <cstdint>
#include <cstdlib>
#include <map>
#include <vector>

#include "../../genedex_b200/csrc/cuda_owners.h"

namespace {
enum Kind { kDev, kPinned, kEvent, kStream, kAsync };
std::map<void *, int> g_live;           // resource -> kind
std::map<void *, void *> g_async_stream;  // async block -> stream it was allocated on
std::vector<uint64_t> g_sizes;          // sizes asked for by every allocating call, in order
std::vector<void *> g_async_freed_on;   // stream of every cudaFreeAsync, in order
uint64_t g_calls = 0, g_fail_at = 0, g_max_bytes = ~0ull, g_bad_frees = 0;

bool fails(uint64_t bytes) { return ++g_calls == g_fail_at || bytes > g_max_bytes; }

cudaError_t acquire(void **p, uint64_t bytes, Kind k) {
    g_sizes.push_back(bytes);
    if (fails(bytes)) {
        *p = (void *)0xdead;  // garbage: an owner must not keep (and later free) what a failed call wrote
        return cudaErrorMemoryAllocation;
    }
    *p = malloc(bytes ? bytes : 1);
    g_live[*p] = k;
    return cudaSuccess;
}

cudaError_t drop(void *p, Kind k) {
    auto it = g_live.find(p);
    if (it == g_live.end() || it->second != k) {
        ++g_bad_frees;
        return cudaErrorInvalidValue;
    }
    g_live.erase(it);
    free(p);
    return cudaSuccess;
}
}  // namespace

// ---- the runtime, as far as the owners use it ------------------------------------------------------------------------
cudaError_t cudaMalloc(void **p, size_t bytes) { return acquire(p, bytes, kDev); }
cudaError_t cudaFree(void *p) { return drop(p, kDev); }
cudaError_t cudaMallocHost(void **p, size_t bytes) { return acquire(p, bytes, kPinned); }
cudaError_t cudaFreeHost(void *p) { return drop(p, kPinned); }
cudaError_t cudaMallocAsync(void **p, size_t bytes, cudaStream_t st) {
    const cudaError_t e = acquire(p, bytes, kAsync);
    if (e == cudaSuccess) g_async_stream[*p] = st;
    return e;
}
cudaError_t cudaFreeAsync(void *p, cudaStream_t st) {
    g_async_freed_on.push_back(st);
    if (g_async_stream.count(p) && g_async_stream[p] != st) ++g_bad_frees;  // freed on another stream
    g_async_stream.erase(p);
    return drop(p, kAsync);
}
cudaError_t cudaEventCreateWithFlags(cudaEvent_t *e, unsigned int) { return acquire((void **)e, 0, kEvent); }
cudaError_t cudaEventDestroy(cudaEvent_t e) { return drop(e, kEvent); }
cudaError_t cudaStreamCreateWithFlags(cudaStream_t *s, unsigned int) { return acquire((void **)s, 0, kStream); }
cudaError_t cudaStreamDestroy(cudaStream_t s) { return drop(s, kStream); }

// ---- control and observation -----------------------------------------------------------------------------------------
extern "C" void emul_reset(uint64_t fail_at, uint64_t max_bytes) {
    g_calls = 0;
    g_fail_at = fail_at;
    g_max_bytes = max_bytes;
    g_sizes.clear();
    g_async_freed_on.clear();
}
extern "C" uint64_t emul_live(int kind) {
    uint64_t n = 0;
    for (const auto &r : g_live) n += r.second == kind;
    return n;
}
extern "C" uint64_t emul_bad_frees() { return g_bad_frees; }
extern "C" uint64_t emul_sizes(uint64_t *out, uint64_t cap) {
    for (uint64_t i = 0; i < g_sizes.size() && i < cap; ++i) out[i] = g_sizes[i];
    return g_sizes.size();
}
extern "C" uint64_t emul_async_frees(void **out, uint64_t cap) {
    for (uint64_t i = 0; i < g_async_freed_on.size() && i < cap; ++i) out[i] = g_async_freed_on[i];
    return g_async_freed_on.size();
}
extern "C" int emul_cuda_free(void *p) { return cudaFree(p); }

// ---- the owners, one handle per heap-allocated owner ------------------------------------------------------------------
#define OWNER_API(T, name)                                                                           \
    extern "C" T *name##_new() { return new T(); }                                                   \
    extern "C" void name##_delete(T *o) { delete o; }                                                \
    extern "C" T *name##_move_new(T *src) { return new T(std::move(*src)); }                         \
    extern "C" void name##_move_assign(T *dst, T *src) { *dst = std::move(*src); }
OWNER_API(gdx::DevMem, dev)
OWNER_API(gdx::HBuf, pinned)
OWNER_API(gdx::AsyncMem, async)
OWNER_API(gdx::Event, event)
OWNER_API(gdx::Stream, stream)

extern "C" int dev_alloc(gdx::DevMem *o, uint64_t n) { return o->alloc(n); }
extern "C" int dev_reserve(gdx::DevMem *o, uint64_t n) { return o->reserve(n); }
extern "C" void dev_reset(gdx::DevMem *o) { o->reset(); }
extern "C" void *dev_release(gdx::DevMem *o) { return o->release(); }
extern "C" void *dev_ptr(gdx::DevMem *o) { return o->p; }
extern "C" uint64_t dev_bytes(gdx::DevMem *o) { return o->bytes; }
extern "C" gdx::DevMem *dev_adopt(void *p, uint64_t n) { return new gdx::DevMem(p, n); }

extern "C" int pinned_alloc(gdx::HBuf *o, uint64_t n) { return o->alloc(n); }
extern "C" int pinned_reserve(gdx::HBuf *o, uint64_t n) { return o->reserve(n); }
extern "C" void *pinned_ptr(gdx::HBuf *o) { return o->p; }
extern "C" uint64_t pinned_bytes(gdx::HBuf *o) { return o->bytes; }

extern "C" int async_alloc(gdx::AsyncMem *o, uint64_t n, void *st) { return o->alloc(n, (cudaStream_t)st); }
extern "C" int async_free(gdx::AsyncMem *o) { return o->free(); }
extern "C" void *async_ptr(gdx::AsyncMem *o) { return o->p; }

extern "C" int event_create(gdx::Event *o) { return o->create(cudaEventDisableTiming); }
extern "C" void *event_handle(gdx::Event *o) { return (cudaEvent_t)*o; }
extern "C" int stream_create(gdx::Stream *o) { return o->create(cudaStreamNonBlocking); }
extern "C" void *stream_handle(gdx::Stream *o) { return (cudaStream_t)*o; }
