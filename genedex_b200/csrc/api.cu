// api.cu -- C ABI of genedex_b200 (include/genedex_b200.h): index handles, device image
// construction from host parts, chunked H2D / kernel / D2H pipelines, locate CSR plumbing.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <type_traits>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstddef>
#include <deque>
#include <thread>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <shared_mutex>
#include <new>
#include <numeric>
#include <string>
#include <utility>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>

#include "../../include/genedex_b200.h"
#include "accel_policy.h"
#include "chunk_plan.h"
#include "cuda_owners.h"
#include "device_build.h"
#include "device_index.h"
#include "host_build.h"
#include "host_pack.h"
#include "kernels.cuh"

using namespace gdx;

// ---- thread-local error / stats state ----------------------------------------------------------------
namespace {

thread_local std::string t_error;
thread_local uint64_t t_error_query = 0;
thread_local gdx_stats t_stats = {};

gdx_status fail(gdx_status st, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    t_error = buf;
    return st;
}

#define CUDA_TRY(expr)                                                                           \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            cudaGetLastError(); /* a failed allocation must not fail the next call's error check */ \
            return fail(_e == cudaErrorMemoryAllocation ? GDX_ERR_OOM : GDX_ERR_CUDA,            \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,        \
                        __LINE__);                                                               \
        }                                                                                        \
    } while (0)

#define GDX_TRY(expr)                  \
    do {                               \
        gdx_status _s = (expr);        \
        if (_s != GDX_OK) return _s;   \
    } while (0)

// exceptions must not cross the C boundary (std::bad_alloc from a host vector, std::system_error from a thread)
template <class F>
gdx_status guarded(F &&f) noexcept {
    try {
        return f();
    } catch (const std::bad_alloc &) {
        return fail(GDX_ERR_OOM, "out of host memory");
    } catch (const std::exception &e) {
        return fail(GDX_ERR_BAD_ARG, "unexpected failure: %s", e.what());
    } catch (...) {
        return fail(GDX_ERR_BAD_ARG, "unexpected failure");
    }
}

uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }
uint64_t div_up(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// The device-resident entry points take their scratch from the stream-ordered pool: keep freed blocks
// cached across synchronisation points instead of returning them to the driver.  Applied once per
// device, with that device current.
void apply_device_settings(int dev) {
    static std::mutex mu;
    static bool done[64] = {};
    if (dev < 0 || dev >= 64) return;
    std::lock_guard<std::mutex> lk(mu);
    if (done[dev]) return;
    done[dev] = true;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        if (dev >= 0 && dev != prev) {
            if (cudaSetDevice(dev) != cudaSuccess) return;
        }
        apply_device_settings(dev >= 0 ? dev : prev);
        ok = true;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// true for cudaMallocHost / cudaHostRegister'ed / managed memory, false for ordinary (pageable) host memory
bool is_pinned(const void *p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
}

uint64_t env_bytes(const char *name, uint64_t dflt) {
    const char *e = getenv(name);
    return e && *e ? (uint64_t)strtoull(e, nullptr, 10) : dflt;
}
// smaller transfers go through the driver's own staging (GDX_STAGE_MIN_BYTES: tests force the staged paths)
const uint64_t kStageMinBytes = env_bytes("GDX_STAGE_MIN_BYTES", 4ull << 20);

constexpr int kSlots = 3;
// Pipeline chunking (defaults 4 / 32 / 4 MB, profiles/r1_ab_pipeline_chunks.txt; the schedule is gdx::ChunkPlan): large
// launches give less launch overhead and deeper shared suffixes for the per-chunk query sort.
uint64_t env_mb(const char *name, uint64_t dflt) {
    const char *e = getenv(name);
    return (uint64_t)(e && atoi(e) > 0 ? atoi(e) : dflt) << 20;
}
const uint64_t kChunkFirst = env_mb("GDX_CHUNK_FIRST_MB", 4);
const uint64_t kChunkMax = env_mb("GDX_CHUNK_MAX_MB", 32);
const uint64_t kChunkTail = env_mb("GDX_CHUNK_TAIL_MB", 4);
constexpr uint64_t kChunkMaxQueries = 64ull << 20;

// (begin, end) event pairs around the kernels of the current call, created on first use and kept for later calls
struct EventPairs {
    struct Pair {
        cudaEvent_t begin, end;
    };
    std::vector<Event> ev;
    size_t used = 0;
    cudaEvent_t take() {
        if (used == ev.size()) {
            Event e;
            if (e.create(cudaEventDefault) != cudaSuccess) return nullptr;  // recording on nullptr fails loudly later
            ev.push_back(std::move(e));
        }
        return ev[used++];
    }
    Pair next() { return Pair{take(), take()}; }
    // the kernel time of every completed pair of the call
    double elapsed_ms() const {
        double ms = 0;
        for (size_t i = 0; i + 1 < used; i += 2) {
            float t = 0;
            cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
            ms += t;
        }
        return ms;
    }
    void reset() { used = 0; }
};

// SA intervals -> hits on one stream.  count() writes the width of every interval, their exclusive scan (the CSR
// offsets, n + 1 entries) and sends the hit total and the number of wide intervals to the pinned words; expand_walk()
// then lists the rows of every interval (wide ones through a worklist) and walks them to text positions.
struct IntervalHits {
    DevMem counts, offsets, scan_tmp, rows, hits, wide;
    struct DeviceWords {
        unsigned long long wide, cursor;  // intervals wider than kExpandInline, worklist cursor
    };
    struct HostWords {
        uint64_t hits, wide;  // pinned: hit total, intervals wider than kExpandInline
    };
    DevMem d_words;
    HBuf h_words;
    Event ev_total;     // *h() is on the host
    EventPairs timing;  // around the locate kernels of the current call
    bool init() {
        return d_words.alloc(sizeof(DeviceWords)) == cudaSuccess && h_words.alloc(sizeof(HostWords)) == cudaSuccess &&
               ev_total.create(cudaEventDisableTiming) == cudaSuccess;
    }
    DeviceWords *d() const { return d_words.as<DeviceWords>(); }
    HostWords *h() const { return h_words.as<HostWords>(); }
    gdx_status count(cudaStream_t st, const uint64_t *starts, const uint64_t *ends, uint64_t n);
    gdx_status expand_walk(const gdx_index *idx, cudaStream_t st, const uint64_t *starts, const uint64_t *ends, uint64_t n,
                           uint64_t n_hits, uint64_t n_wide, unsigned long long *walk_steps, bool hit32);
};

struct Slot {
    Stream stream;
    DevMem bytes, offsets, out_a, out_b, sort;
    IntervalHits locate;  // pipelined locate: the chunk's CSR, rows and hits
    // staging for pageable caller buffers / packed queries / narrow results
    HBuf h_in, h_off, h_out_a, h_out_b;
    // queries of a packed chunk that hold a byte without a 2-bit code: offsets + slots + IO bytes, re-run raw
    HBuf h_x;
    DevMem xbuf;
    Event ev_h2d, ev_out;
    Event ev_link;  // the chunk's query upload has left the PCIe link
    bool h2d_pending = false;
    EventPairs timing;  // around the search kernels of the current call
};

// The words one call shares with its kernels, in pinned host memory and on the device.  Error words hold the smallest
// failing index (atomicMin), kNoError if there is none; the counters are sums (atomicAdd).
struct Counters {
    uint64_t err[kSlots];         // k_search per slot stream; k_hamming pass 1 on slot 0
    uint64_t extend_bad_symbol;   // k_extend: err[0]
    uint64_t extend_bad_cursor;   // k_extend: err[1]
    SearchCounters search;        // k_search
    unsigned long long locate_walk_steps;   // k_locate_walk, k_locate_walk_compact
    unsigned long long hamming_expansions;  // k_hamming pass 1
};
static_assert(offsetof(Counters, extend_bad_cursor) == offsetof(Counters, extend_bad_symbol) + 8,
              "k_extend reports a bad cursor in the word after its error word");

struct Workspace {
    Slot slot[kSlots];
    HBuf cnt_host;
    DevMem cnt_dev;
    DevMem starts, ends, symbols;
    IntervalHits locate;  // gdx_locate_intervals and the Hamming locate
    Event ev_a;           // orders the slot streams behind the reset of the counters (search_host)
    Counters *cnt_h() const { return cnt_host.as<Counters>(); }  // pinned
    Counters *cnt_d() const { return cnt_dev.as<Counters>(); }   // device
    // error words to kNoError, counters to zero
    cudaError_t reset_counters(cudaStream_t st) {
        constexpr size_t kErrBytes = offsetof(Counters, search);
        const cudaError_t e = cudaMemsetAsync(cnt_d(), 0xff, kErrBytes, st);
        return e != cudaSuccess ? e : cudaMemsetAsync((uint8_t *)cnt_d() + kErrBytes, 0, sizeof(Counters) - kErrBytes, st);
    }
    cudaError_t read_counters(cudaStream_t st) {
        return cudaMemcpyAsync(cnt_h(), cnt_d(), sizeof(Counters), cudaMemcpyDeviceToHost, st);
    }
    void reset_timing() {
        for (auto &s : slot) {
            s.timing.reset();
            s.locate.timing.reset();
        }
        locate.timing.reset();
    }
};

// a workspace with its streams, events and words, or nullptr when one of them cannot be created
std::unique_ptr<Workspace> new_workspace() {
    auto w = std::make_unique<Workspace>();
    for (auto &s : w->slot)
        if (s.stream.create(cudaStreamNonBlocking) != cudaSuccess || !s.locate.init() ||
            s.ev_h2d.create(cudaEventDisableTiming) != cudaSuccess || s.ev_out.create(cudaEventDisableTiming) != cudaSuccess ||
            s.ev_link.create(cudaEventDisableTiming) != cudaSuccess)
            return nullptr;
    if (w->cnt_host.alloc(sizeof(Counters)) != cudaSuccess || w->cnt_dev.alloc(sizeof(Counters)) != cudaSuccess ||
        !w->locate.init() || w->ev_a.create(cudaEventDefault) != cudaSuccess)
        return nullptr;
    return w;
}

// a pinned hit buffer of the index, lent to one call at a time
struct PinnedHits {
    HBuf buf;
    bool in_use = false;
};

}  // namespace

struct gdx_index {
    ImageHeader h;
    void *image = nullptr;
    DevMem owned_image;            // holds image unless it was adopted with own_image = 0
    int device = 0;
    DevIndex dev;                  // written by refresh_dev only
    // accelerators outside the image (gdx_index_set_dense_suffix_array / _seed_table_depth / _row_context_table)
    DevMem dense_sa, seed_table, row_context, compact_seed;
    uint32_t seed_depth = 0, compact_depth = 0;
    bool verify = true;            // finish one-row intervals through the text section (gdx_index_set_text_verification)
    PackTable pack;                // io byte -> 2-bit code (host packer, host_pack.h)
    // host-buffer queries hold this shared for the whole call; (re)building or freeing an accelerator needs it
    // exclusively and reports GDX_ERR_BUSY instead of pulling memory from under a running kernel
    mutable std::shared_mutex cfg_mu;
    mutable std::mutex mu;
    mutable std::vector<std::unique_ptr<Workspace>> free_ws;
    mutable std::vector<PinnedHits> pinned;
};

namespace {

std::unique_ptr<Workspace> acquire_ws(const gdx_index *idx) {
    {
        std::lock_guard<std::mutex> lk(idx->mu);
        if (!idx->free_ws.empty()) {
            std::unique_ptr<Workspace> w = std::move(idx->free_ws.back());
            idx->free_ws.pop_back();
            return w;
        }
    }
    return new_workspace();
}
struct WsLease {
    const gdx_index *idx;
    std::unique_ptr<Workspace> w;
    explicit WsLease(const gdx_index *i) : idx(i), w(acquire_ws(i)) {}
    ~WsLease() {
        if (!w) return;
        std::lock_guard<std::mutex> lk(idx->mu);
        idx->free_ws.push_back(std::move(w));
    }
};

// a failed call must not return while one of its streams still reads or writes the caller's buffers; the error that
// made it fail stays the reported one
void drain(Workspace *ws) {
    for (int s = 0; s < kSlots; ++s) cudaStreamSynchronize(ws->slot[s].stream);
    cudaGetLastError();
}

// runs f(ws) on a workspace leased for one host-buffer call, with the configuration held shared and idx's device
// current; drains the workspace when f fails
template <class F>
gdx_status with_workspace(const gdx_index *idx, F &&f) {
    std::shared_lock<std::shared_mutex> cfg(idx->cfg_mu);
    DeviceGuard guard(idx->device);
    WsLease lease(idx);
    if (!lease.w) return fail(GDX_ERR_CUDA, "could not create a CUDA workspace: %s", cudaGetErrorString(cudaGetLastError()));
    lease.w->reset_timing();
    const gdx_status st = f(lease.w.get());
    if (st != GDX_OK) drain(lease.w.get());
    return st;
}

// runs f() with the configuration of idx held exclusively and idx's device current; busy is the GDX_ERR_BUSY message
// while host-buffer queries hold the configuration
template <class F>
gdx_status with_config(gdx_index *idx, const char *busy, F &&f) {
    return guarded([&]() -> gdx_status {
        if (!idx) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        std::unique_lock<std::shared_mutex> cfg(idx->cfg_mu, std::try_to_lock);
        if (!cfg.owns_lock()) return fail(GDX_ERR_BUSY, "%s", busy);
        DeviceGuard guard(idx->device);
        return f();
    });
}

// ---- layout dispatch -----------------------------------------------------------------------------------
template <class F>
gdx_status dispatch_layout(const RankLayout &L, F &&f) {
    if (L.kind == kLayoutK32) return f(K32{});
    switch (L.planes) {
    case 1: return f(KG<1>{});
    case 2: return f(KG<2>{});
    case 3: return f(KG<3>{});
    case 4: return f(KG<4>{});
    case 5: return f(KG<5>{});
    case 6: return f(KG<6>{});
    case 7: return f(KG<7>{});
    case 8: return f(KG<8>{});
    }
    return fail(GDX_ERR_UNSUPPORTED, "unsupported number of bit planes %u", L.planes);
}

// ---- device image construction -------------------------------------------------------------------------
// u32 or u64 words on the host or on the device (at most one of the pointers is set)
struct Words {
    const uint64_t *h64 = nullptr;
    const uint32_t *h32 = nullptr;
    const void *d = nullptr;
    bool d_wide = false;
    bool any() const { return h64 || h32 || d; }
};

struct ImageSources {
    const gdx_alphabet *alphabet;
    uint32_t storage, sampling_rate, lookup_depth;
    uint64_t n;
    const uint64_t *count;             // host, sigma + 1
    const uint64_t *sentinels;         // host
    uint64_t ntexts;
    const uint64_t *border_rows;       // host, sorted ascending together with border_pos
    const uint64_t *border_pos;        // host
    uint64_t n_border;
    const uint8_t *d_bwt;              // device, n bytes
    const uint8_t *d_text = nullptr;   // device, n bytes dense text (optional: enables the text section)
    Words samples;                     // the sampled suffix array (set when n > 0)
    Words isa;                         // optional sampled inverse suffix array, only together with d_text
    // accelerator policy of the index (travels with the image)
    uint32_t accel_flags = 0;
    uint64_t accel_budget = 0;
};

uint32_t accel_flags_from_config(uint32_t flags) {
    return ((flags & GDX_FLAG_NO_DENSE_SUFFIX_ARRAY) ? kAccelNoDenseSA : 0u) |
           ((flags & GDX_FLAG_NO_SEED_TABLE) ? kAccelNoSeedTable : 0u) |
           ((flags & GDX_FLAG_NO_ROW_CONTEXT_TABLE) ? kAccelNoRowContext : 0u);
}

gdx_status validate_alphabet(const gdx_alphabet &a) {
    if (a.num_dense_symbols < 2 || a.num_dense_symbols > 256)
        return fail(GDX_ERR_BAD_ARG, "alphabet size must be in [2,256] incl. the sentinel (alphabet.rs:166-174)");
    if (a.num_searchable_dense_symbols < 1 || a.num_searchable_dense_symbols > a.num_dense_symbols - 1)
        return fail(GDX_ERR_BAD_ARG, "there must be at least one searchable symbol (alphabet.rs:186-189)");
    for (int i = 0; i < 256; ++i)
        if (a.io_to_dense[i] >= a.num_dense_symbols)
            return fail(GDX_ERR_BAD_ARG, "io_to_dense[%d] = %u is not a dense symbol", i, a.io_to_dense[i]);
    return GDX_OK;
}

// wide_override: -1 = decide from the text length (and GDX_FORCE_WIDE), 0 / 1 = as given (header validation)
gdx_status plan_header(const ImageSources &src, ImageHeader &h, int wide_override = -1) {
    memset(&h, 0, sizeof h);
    h.magic = kImageMagic;
    h.version = GDX_ABI_VERSION;
    h.n = src.n;
    h.ntexts = src.ntexts;
    h.n_border = src.n_border;
    h.sigma = src.alphabet->num_dense_symbols;
    h.ns = src.alphabet->num_searchable_dense_symbols;
    h.storage = src.storage;
    h.sampling_rate = src.sampling_rate;
    h.lookup_depth = src.lookup_depth;
    h.accel_flags = src.accel_flags;
    h.accel_budget = src.accel_budget;
    // 64-bit samples / lookup entries are only needed beyond 2^32 - 1 symbols; GDX_FORCE_WIDE=1 selects them
    // for any text so that this path can be tested without a 4.3 G symbol index
    const char *fw = getenv("GDX_FORCE_WIDE");
    h.wide = (src.n > 0xffffffffull || (fw && atoi(fw) != 0)) ? 1 : 0;
    if (wide_override >= 0) h.wide = (src.n > 0xffffffffull || wide_override) ? 1 : 0;
    h.layout = choose_layout(h.sigma);
    memcpy(h.io_to_dense, src.alphabet->io_to_dense, 256);
    if (src.lookup_depth > kMaxLookupDepth)
        return fail(GDX_ERR_UNSUPPORTED, "lookup table depth %u > %u", src.lookup_depth, kMaxLookupDepth);
    const uint64_t P = 1ull << h.layout.log2_pos;
    h.n_records = div_up(src.n + 1, P);
    h.n_superblocks = div_up(src.n + 1, 1ull << kSuperblockLog2);
    h.n_samples = div_up(src.n, src.sampling_rate);
    uint64_t entries = 0, pw = 1;
    for (uint32_t d = 0; d <= kMaxLookupDepth; ++d) {
        h.lut_level_off[d] = entries;
        h.lut_pow[d] = pw;
        if (d <= src.lookup_depth) {
            entries += pw;
            if (entries > (1ull << 36) || pw > (1ull << 36))
                return fail(GDX_ERR_UNSUPPORTED, "lookup tables of depth %u are too large", src.lookup_depth);
            pw *= h.ns;
        }
    }
    const uint64_t esz = h.wide ? 8 : 4;
    uint64_t off = 0;
    auto place = [&](uint64_t bytes) {
        uint64_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    h.off_records = place(h.n_records * h.layout.stride);
    // pack kernels write totals for whole superblock CTAs
    h.off_sbc = place(h.n_superblocks * h.layout.noff * 8);
    h.off_samples = place(h.n_samples * esz);
    h.off_lookup = place(entries * 2 * esz);
    h.off_border_rows = place(h.n_border * 8);
    h.off_border_pos = place(h.n_border * 8);
    h.off_sentinels = place(h.ntexts * 8);
    h.off_count = place((uint64_t)(h.sigma + 1) * 8);
    h.text_bits = 0;
    h.off_text = off;
    if (src.d_text) {
        h.text_bits = h.sigma <= 16 ? 4 : 8;
        // + 16: the comparison reads whole 64-bit words, one past the last (compare_with_text)
        h.off_text = place((h.text_bits == 4 ? (src.n + 1) / 2 : src.n) + 16);
    }
    h.has_isa = 0;
    h.off_isa = off;
    if (h.text_bits && src.isa.any()) {
        h.has_isa = 1;
        h.off_isa = place(h.n_samples * esz);
    }
    h.image_bytes = off;
    return GDX_OK;
}

// An image header that comes from a file or a peer is untrusted: every size, offset and the record layout are
// re-derived from its scalar fields and must match, so that no kernel ever indexes with a value the planner
// would not have produced.
gdx_status validate_header(const ImageHeader &h) {
    if (h.magic != kImageMagic || h.version != GDX_ABI_VERSION)
        return fail(GDX_ERR_BAD_ARG, "not a genedex_b200 image header of this version (magic/version mismatch)");
    gdx_alphabet a;
    memcpy(a.io_to_dense, h.io_to_dense, 256);
    a.num_dense_symbols = h.sigma;
    a.num_searchable_dense_symbols = h.ns;
    GDX_TRY(validate_alphabet(a));
    if (h.sampling_rate == 0 || h.lookup_depth > kMaxLookupDepth || h.storage > GDX_I64 || h.ntexts == 0 ||
        h.n_border > h.n || h.ntexts > h.n || (h.text_bits != 0 && h.text_bits != 4 && h.text_bits != 8) || h.has_isa > 1 ||
        h.wide > 1 || h.n > (1ull << 48))
        return fail(GDX_ERR_BAD_ARG, "image header: field out of range");
    ImageSources src;
    src.alphabet = &a;
    src.storage = h.storage;
    src.sampling_rate = h.sampling_rate;
    src.lookup_depth = h.lookup_depth;
    src.n = h.n;
    src.ntexts = h.ntexts;
    src.n_border = h.n_border;
    src.d_text = h.text_bits ? reinterpret_cast<const uint8_t *>(&a) : nullptr;            // presence only
    src.isa.d = h.has_isa ? &a : nullptr;                                                 // presence only
    src.accel_flags = h.accel_flags;
    src.accel_budget = h.accel_budget;
    ImageHeader want;
    GDX_TRY(plan_header(src, want, (int)h.wide));
    if (memcmp(&want, &h, sizeof(ImageHeader)) != 0)
        return fail(GDX_ERR_BAD_ARG, "image header is inconsistent (sizes / offsets do not match its own fields)");
    return GDX_OK;
}

// ---- accelerators outside the image (include/genedex_b200.h, policy in accel_policy.h) ---------------------
bool verify_enabled();

// idx->dev from the image and the accelerators the index holds; nothing else writes idx->dev
void refresh_dev(gdx_index *idx) {
    DevIndex d = make_dev_index(idx->h, idx->image);
    if (idx->dense_sa) {  // resolve_row / k_locate_walk see a suffix array with sampling rate 1
        d.samples = idx->dense_sa.p;
        d.sampling_rate = 1;
        d.sampling_shift = 0;
    }
    if (idx->seed_table) {
        d.seed_lookup = idx->seed_table.p;
        d.seed_depth = idx->seed_depth;
    }
    d.row_context = idx->row_context.p;
    if (idx->compact_seed) {
        d.compact_seed = idx->compact_seed.as<uint8_t>();
        d.compact_pool = reinterpret_cast<const uint32_t *>(
            d.compact_seed + cs_groups(seed_entries(idx->h.ns, idx->compact_depth)) * kCsGroupBytes);
        d.compact_depth = idx->compact_depth;
    }
    d.verify_min_remaining = verify_min_remaining((bool)idx->dense_sa, getenv("GDX_VERIFY_MIN"));
    idx->dev = d;
}

gdx_status table_oom(const char *what, uint64_t bytes) {
    cudaGetLastError();
    return fail(GDX_ERR_OOM, "%s: %llu bytes of device memory not available", what, (unsigned long long)bytes);
}

// table := `bytes` of device memory filled by launch(L, p) for the rank layout L of the index, once the kernel is done
template <class F>
gdx_status fill_table(gdx_index *idx, DevMem &table, uint64_t bytes, const char *what, F &&launch) {
    DevMem d;
    if (d.alloc(bytes) != cudaSuccess) return table_oom(what, bytes);
    GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
        launch(L, d.p);
        return GDX_OK;
    }));
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    table = std::move(d);
    refresh_dev(idx);
    return GDX_OK;
}

void drop_table(gdx_index *idx, DevMem &table) {
    table = DevMem();
    refresh_dev(idx);
}

AccelPolicy accel_policy(const ImageHeader &h) {
    return AccelPolicy{h.n, h.accel_budget, h.ns, h.lookup_depth, h.wide != 0, h.text_bits != 0,
                       (h.accel_flags & kAccelNoDenseSA) != 0, (h.accel_flags & kAccelNoSeedTable) != 0,
                       (h.accel_flags & kAccelNoRowContext) != 0};
}

gdx_status build_dense_sa(gdx_index *idx) {
    if (idx->dense_sa || idx->h.n == 0) return GDX_OK;
    const uint64_t n = idx->h.n;
    return fill_table(idx, idx->dense_sa, n * (idx->h.wide ? 8 : 4), "dense suffix array", [&](auto L, void *d) {
        k_densify<decltype(L)><<<(unsigned)div_up(n, 256), 256>>>(idx->dev, d, n);
    });
}

gdx_status build_row_context(gdx_index *idx) {
    if (idx->row_context) return GDX_OK;
    if (!accel_policy(idx->h).row_context_possible())
        return fail(GDX_ERR_UNSUPPORTED, "the row context table needs the text section, at most 4 searchable symbols and a "
                                         "text shorter than 2^32 symbols");
    const uint64_t n = idx->h.n;
    return fill_table(idx, idx->row_context, n * 16, "row context table", [&](auto L, void *d) {
        k_build_row_context<decltype(L)><<<(unsigned)div_up(n, 256), 256>>>(idx->dev, reinterpret_cast<uint4 *>(d), n);
    });
}

// count words to dst as u64 (wide) or u32, converted on the host or on the device where the source has the other width
cudaError_t put_words(void *dst, uint64_t count, bool wide, const Words &w) {
    const uint64_t esz = wide ? 8 : 4;
    if (w.d && w.d_wide == wide) return cudaMemcpy(dst, w.d, count * esz, cudaMemcpyDeviceToDevice);
    if (w.d) {
        const unsigned g = (unsigned)div_up(count, 256);
        if (wide) k_widen_u32<<<g, 256>>>((const uint32_t *)w.d, count, (uint64_t *)dst);
        else k_narrow_u64<<<g, 256>>>((const uint64_t *)w.d, count, (uint32_t *)dst);
        return cudaGetLastError();
    }
    if (wide ? w.h64 != nullptr : w.h32 != nullptr)
        return cudaMemcpy(dst, wide ? (const void *)w.h64 : w.h32, count * esz, cudaMemcpyHostToDevice);
    if (!w.any()) return cudaSuccess;
    auto convert = [&](auto zero) {
        std::vector<decltype(zero)> v(count);
        for (uint64_t i = 0; i < count; ++i) v[i] = (decltype(zero))(w.h64 ? w.h64[i] : w.h32[i]);
        return cudaMemcpy(dst, v.data(), count * esz, cudaMemcpyHostToDevice);
    };
    return wide ? convert(uint64_t{}) : convert(uint32_t{});
}

// level 0 of a lookup table: [(0, n)] (lookup_table.rs:205-209)
cudaError_t put_lookup_level0(void *dst, uint64_t n, bool wide) {
    const uint64_t e0[2] = {0, n};
    return put_words(dst, 2, wide, Words{e0});
}

gdx_status build_seed_table(gdx_index *idx, uint32_t depth) {
    drop_table(idx, idx->compact_seed);  // it goes with the seed table
    drop_table(idx, idx->seed_table);
    const ImageHeader &h = idx->h;
    // a level no deeper than the configured table would change nothing for the better and would move the
    // eager translation of the configured suffix (lookup_table.rs:154-157): not built
    if (depth <= h.lookup_depth || h.n == 0 || h.ns == 0) return GDX_OK;
    const uint64_t esz = h.wide ? 16 : 8, last = seed_entries(h.ns, depth), prev = seed_entries(h.ns, depth - 1);
    if (last == 0 || depth > 40) return fail(GDX_ERR_UNSUPPORTED, "seed table of depth %u is too large", depth);
    // levels alternate between the final buffer and a temporary one of the size of level depth - 1
    DevMem fin, tmp;
    if (fin.alloc(last * esz) != cudaSuccess || tmp.alloc(prev * esz) != cudaSuccess) {
        char what[40];
        snprintf(what, sizeof what, "seed table of depth %u", depth);
        return table_oom(what, (last + prev) * esz);
    }
    // level 0 lives where level `depth` will not collide: parity of depth
    void *cur = (depth % 2 == 0) ? fin.p : tmp.p;
    cudaError_t e = put_lookup_level0(cur, h.n, h.wide);
    for (uint32_t d = 1; d <= depth && e == cudaSuccess; ++d) {
        void *nxt = cur == fin.p ? tmp.p : fin.p;
        const uint64_t entries = seed_entries(h.ns, d);
        GDX_TRY(dispatch_layout(h.layout, [&](auto L) -> gdx_status {
            k_lut_extend<decltype(L)><<<(unsigned)div_up(entries, 256), 256>>>(idx->dev, cur, nxt, entries);
            return GDX_OK;
        }));
        e = cudaGetLastError();
        cur = nxt;
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess || cur != fin.p) return fail(GDX_ERR_CUDA, "seed table: %s", cudaGetErrorString(e));
    idx->seed_table = std::move(fin);
    idx->seed_depth = depth;
    refresh_dev(idx);
    return GDX_OK;
}

uint64_t free_device_bytes() {
    size_t free_b = 0, total_b = 0;
    return cudaMemGetInfo(&free_b, &total_b) == cudaSuccess ? free_b : kFreeUnknown;
}

uint64_t accel_bytes(const gdx_index *idx) {
    return idx->dense_sa.bytes + idx->seed_table.bytes + idx->row_context.bytes + idx->compact_seed.bytes;
}

// The compact seed level of depth d (compact_seed.h) from suffix array order and the text section.  A counting pass
// sizes the exception records first; *fits = false (nothing built, no error) when the groups and records do not fit
// what the policy leaves.
gdx_status build_compact_seed_level(gdx_index *idx, uint32_t d, bool *fits) {
    const ImageHeader &h = idx->h;
    const AccelPolicy p = accel_policy(h);
    *fits = false;
    const uint64_t n = h.n, groups = cs_groups(seed_entries(h.ns, d)), group_bytes = groups * kCsGroupBytes;
    const unsigned grid = (unsigned)div_up(n + 1, 256);
    DevMem counters;  // n_exc, order_error
    CUDA_TRY(counters.alloc(16));
    CUDA_TRY(cudaMemset(counters.p, 0, 16));
    CsBuild b{};
    b.n_groups = groups;
    b.d = d;
    b.n_exc = counters.as<unsigned long long>();
    b.order_error = reinterpret_cast<unsigned int *>(counters.as<uint8_t>() + 8);
    auto rows_pass = [&]() -> gdx_status {
        GDX_TRY(dispatch_layout(h.layout, [&](auto L) -> gdx_status {
            k_cs_rows<decltype(L)><<<grid, 256>>>(idx->dev, b);
            return GDX_OK;
        }));
        const cudaError_t e = cudaDeviceSynchronize();
        return e == cudaSuccess ? GDX_OK : fail(GDX_ERR_CUDA, "compact seed level: %s", cudaGetErrorString(e));
    };
    GDX_TRY(rows_pass());
    uint64_t m = 0;
    uint32_t order_error = 0;
    CUDA_TRY(cudaMemcpy(&m, counters.p, 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(&order_error, b.order_error, 4, cudaMemcpyDeviceToHost));
    if (order_error) return fail(GDX_ERR_CUDA, "compact seed level: the rows are not in suffix array order");
    // pool: one count per group with a record (at most one per exception) + a triple per exception
    const uint64_t pool_words = 4 * m;
    if (m >= (1ull << 30) || !p.compact_seed_fits(d, pool_words * 4, accel_bytes(idx), free_device_bytes()))
        return GDX_OK;
    DevMem table, key, val, tmp;
    if (table.alloc(group_bytes + pool_words * 4) != cudaSuccess) return table_oom("compact seed level", group_bytes + pool_words * 4);
    int end_bit = 1;  // d-mer indices are below ns^d
    while (end_bit < 64 && (seed_entries(h.ns, d) >> end_bit) != 0) ++end_bit;
    size_t sort_bytes = 0, scan_bytes = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint64_t *)nullptr, (uint64_t *)nullptr,
                                             (const uint64_t *)nullptr, (uint64_t *)nullptr, (int)m, 0, end_bit));
    CUDA_TRY(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)m));
    const uint64_t piece = align_up(m * 8 + 8, 256);
    if (key.alloc(2 * piece) != cudaSuccess || val.alloc(2 * piece) != cudaSuccess ||
        tmp.alloc(align_up(std::max(sort_bytes, scan_bytes), 256) + 2 * piece) != cudaSuccess)
        return table_oom("compact seed level (build)", 4 * piece + std::max(sort_bytes, scan_bytes));
    uint64_t *key_in = key.as<uint64_t>(), *key_out = (uint64_t *)(key.as<uint8_t>() + piece);
    uint64_t *val_in = val.as<uint64_t>(), *val_out = (uint64_t *)(val.as<uint8_t>() + piece);
    uint32_t *flag = (uint32_t *)tmp.p, *ord = (uint32_t *)(tmp.as<uint8_t>() + piece);
    void *cub_tmp = tmp.as<uint8_t>() + 2 * piece;
    CUDA_TRY(cudaMemset(table.p, 0, group_bytes));
    CUDA_TRY(cudaMemset(counters.p, 0, 8));
    b.groups = table.as<uint8_t>();
    b.write = 1;
    b.exc_cap = m;
    b.exc_key = key_in;
    b.exc_val = val_in;
    GDX_TRY(rows_pass());
    if (m) {
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp, sort_bytes, key_in, key_out, val_in, val_out, (int)m, 0, end_bit));
        const unsigned g = (unsigned)div_up(m, 256);
        k_cs_first_of_group<<<g, 256>>>(key_out, m, flag);
        CUDA_TRY(cub::DeviceScan::InclusiveSum(cub_tmp, scan_bytes, flag, ord, (int)m));
        k_cs_records<<<g, 256>>>(key_out, val_out, ord, m, table.as<uint8_t>(), (uint32_t *)(table.as<uint8_t>() + group_bytes));
        const cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "compact seed level: %s", cudaGetErrorString(e));
    }
    idx->compact_seed = std::move(table);
    idx->compact_depth = d;
    refresh_dev(idx);
    *fits = true;
    return GDX_OK;
}

// the compact seed level of the seed table the index holds now: the deepest level the policy allows whose groups and
// records fit, or none
gdx_status build_compact_seed(gdx_index *idx) {
    drop_table(idx, idx->compact_seed);
    const AccelPolicy p = accel_policy(idx->h);
    const uint32_t seed = idx->seed_table ? idx->seed_depth : 0;
    for (uint32_t d = p.compact_seed_max_depth(seed); d > seed; --d) {
        if (!p.compact_seed_fits(d, 0, accel_bytes(idx), free_device_bytes())) continue;
        bool fits = false;
        GDX_TRY(build_compact_seed_level(idx, d, &fits));
        if (fits) break;
    }
    return GDX_OK;
}

// what the policy of the index allows, in this order; each table is optional, so a failed build is no error of the call
void build_accelerators(gdx_index *idx) {
    const AccelPolicy p = accel_policy(idx->h);
    auto used = [&] { return accel_bytes(idx); };
    if (p.dense_sa(used(), free_device_bytes(), getenv("GDX_DENSE_SA")) && build_dense_sa(idx) != GDX_OK)
        t_error.clear();
    const uint32_t depth = p.seed_depth(used(), free_device_bytes(), getenv("GDX_SEED_TABLE"));
    if (depth && build_seed_table(idx, depth) != GDX_OK) t_error.clear();
    if (p.row_context(used(), free_device_bytes(), getenv("GDX_ROW_CONTEXT")) && build_row_context(idx) != GDX_OK)
        t_error.clear();
    // last: the three tables above build exactly what they would without it
    if (build_compact_seed(idx) != GDX_OK) t_error.clear();
}

// Every way of creating an index ends here, with a finished image.  The caller has the device current and has released
// its device temporaries, so that the policy sees what the index leaves free.  On failure the image stays the caller's.
gdx_status open_index(const ImageHeader &h, void *image, bool own_image, int device, gdx_index **out) {
    gdx_index *idx = new (std::nothrow) gdx_index();
    if (!idx) return fail(GDX_ERR_OOM, "out of host memory");
    idx->h = h;
    idx->image = image;
    if (own_image) idx->owned_image = DevMem(image, h.image_bytes);
    idx->device = device;
    build_pack_table(h.io_to_dense, h.ns, idx->pack);
    idx->verify = verify_enabled();
    refresh_dev(idx);
    build_accelerators(idx);
    *out = idx;
    return GDX_OK;
}

// an image built here: the index owns it once it is open
gdx_status open_index(const ImageHeader &h, DevMem &image, int device, gdx_index **out) {
    GDX_TRY(open_index(h, image.p, true, device, out));
    image.release();
    return GDX_OK;
}

// the host BWT (n bytes) on the device
gdx_status upload_bwt(const uint8_t *bwt, uint64_t n, DevMem &d_bwt) {
    CUDA_TRY(d_bwt.alloc(n));
    const cudaError_t e = cudaMemcpy(d_bwt.p, bwt, n, cudaMemcpyHostToDevice);
    return e == cudaSuccess ? GDX_OK : fail(GDX_ERR_CUDA, "BWT upload failed: %s", cudaGetErrorString(e));
}

// fills h and a new image from src; the caller releases its temporaries and then opens the index over the image
gdx_status build_image(const ImageSources &src, ImageHeader &h, DevMem &image) {
    GDX_TRY(plan_header(src, h));
    CUDA_TRY(image.alloc(h.image_bytes));
    uint8_t *base = image.as<uint8_t>();
    CUDA_TRY(cudaMemset(base, 0, h.image_bytes));
    CUDA_TRY(cudaMemcpy(base + h.off_sentinels, src.sentinels, h.ntexts * 8, cudaMemcpyHostToDevice));
    if (h.n_border) {
        CUDA_TRY(cudaMemcpy(base + h.off_border_rows, src.border_rows, h.n_border * 8, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(base + h.off_border_pos, src.border_pos, h.n_border * 8, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMemcpy(base + h.off_count, src.count, (uint64_t)(h.sigma + 1) * 8, cudaMemcpyHostToDevice));

    // rank records + superblock table
    uint64_t *sbc = (uint64_t *)(base + h.off_sbc);
    if (h.layout.kind == kLayoutK32) {
        k_pack_k32<<<(unsigned)h.n_superblocks, 1024>>>(src.d_bwt, h.n, h.layout.noff, base + h.off_records,
                                                        h.n_records, sbc);
    } else {
        GDX_TRY(dispatch_layout(h.layout, [&](auto L) -> gdx_status {
            using LT = decltype(L);
            if constexpr (!std::is_same<LT, K32>::value) {
                constexpr int B = LT::kPlanes;
                k_pack_kg<B><<<(unsigned)h.n_superblocks, 512>>>(src.d_bwt, h.n, h.sigma, h.layout.stride,
                                                                 base + h.off_records, h.n_records, sbc);
            }
            return GDX_OK;
        }));
    }
    CUDA_TRY(cudaGetLastError());
    k_sb_scan<<<div_up(h.layout.noff, 64), 64>>>(sbc, h.n_superblocks, h.layout.noff,
                                                 (const uint64_t *)(base + h.off_count));
    CUDA_TRY(cudaGetLastError());

    if (h.n_samples) CUDA_TRY(put_words(base + h.off_samples, h.n_samples, h.wide, src.samples));
    if (h.has_isa && h.n_samples) CUDA_TRY(put_words(base + h.off_isa, h.n_samples, h.wide, src.isa));
    if (h.text_bits && h.n) {
        const uint64_t items = h.text_bits == 4 ? (h.n + 1) / 2 : h.n;
        k_pack_text<<<(unsigned)div_up(items, 256), 256>>>(src.d_text, h.n, h.text_bits, base + h.off_text);
        CUDA_TRY(cudaGetLastError());
    }

    // lookup tables: level d from level d-1
    const DevIndex dev = make_dev_index(h, base);
    void *lut = base + h.off_lookup;
    CUDA_TRY(put_lookup_level0(lut, h.n, h.wide));
    for (uint32_t d = 1; d <= h.lookup_depth; ++d) {
        GDX_TRY(dispatch_layout(h.layout, [&](auto L) -> gdx_status {
            k_lut_fill<decltype(L)><<<(unsigned)div_up(h.lut_pow[d], 256), 256>>>(dev, lut, d);
            return GDX_OK;
        }));
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaDeviceSynchronize());
    return GDX_OK;
}

gdx_status check_text_offsets(const uint64_t *text_offsets, uint64_t num_texts) {
    for (uint64_t i = 0; i < num_texts; ++i)
        if (text_offsets[i + 1] < text_offsets[i])
            return fail(GDX_ERR_BAD_ARG, "text_offsets must be non-decreasing (text %llu)", (unsigned long long)i);
    return GDX_OK;
}

gdx_status check_config(const gdx_config &c) {
    if (c.suffix_array_sampling_rate == 0)
        return fail(GDX_ERR_BAD_ARG, "suffix array sampling rate must be > 0 (config.rs:28)");
    if (c.storage > GDX_I64) return fail(GDX_ERR_BAD_ARG, "unknown index storage %u", c.storage);
    if (c.construction > GDX_CONSTRUCT_AUTO) return fail(GDX_ERR_BAD_ARG, "unknown construction mode %u", c.construction);
    return GDX_OK;
}

gdx_status resolve_device(int32_t requested, int *device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(GDX_ERR_CUDA, "no CUDA device available: %s (genedex_b200 has no CPU fallback)",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (requested < 0) {
        CUDA_TRY(cudaGetDevice(device));
    } else {
        if (requested >= count) return fail(GDX_ERR_BAD_ARG, "device %d out of range (%d devices)", requested, count);
        *device = requested;
    }
    return GDX_OK;
}

}  // namespace

// ================================================================================================
// misc
// ================================================================================================
extern "C" uint32_t gdx_abi_version(void) { return GDX_ABI_VERSION; }
extern "C" const char *gdx_last_error_message(void) { return t_error.c_str(); }
extern "C" uint64_t gdx_last_error_query(void) { return t_error_query; }
extern "C" int32_t gdx_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) return 0;
    return c;
}
extern "C" gdx_status gdx_get_stats(gdx_stats *out) {
    if (!out) return fail(GDX_ERR_BAD_ARG, "out is NULL");
    *out = t_stats;
    return GDX_OK;
}
extern "C" uint32_t gdx_host_pool_resize(uint32_t threads) {
    try {
        return HostPool::get().resize(threads);
    } catch (...) {  // (a thread could not be started: the pool keeps the workers it has)
        return HostPool::get().threads();
    }
}
extern "C" void gdx_host_pack_tuning(int32_t prefetch_bytes, int32_t streaming_stores) { set_pack_tuning(prefetch_bytes, streaming_stores); }
extern "C" gdx_status gdx_host_alloc(uint64_t bytes, void **out) {
    if (!out) return fail(GDX_ERR_BAD_ARG, "out is NULL");
    CUDA_TRY(cudaMallocHost(out, bytes ? bytes : 1));
    return GDX_OK;
}
extern "C" void gdx_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// ================================================================================================
// construction
// ================================================================================================
extern "C" gdx_status gdx_index_build(const uint8_t *texts, const uint64_t *text_offsets, uint64_t num_texts,
                                      const gdx_alphabet *alphabet, const gdx_config *config, gdx_index **out) {
    return guarded([&]() -> gdx_status {
        if (!out) return fail(GDX_ERR_BAD_ARG, "out is NULL");
        *out = nullptr;
        if (!text_offsets || !alphabet || !config) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        if (num_texts == 0) return fail(GDX_ERR_BAD_ARG, "there should be at least one text (construction/mod.rs:300)");
        GDX_TRY(check_text_offsets(text_offsets, num_texts));
        GDX_TRY(validate_alphabet(*alphabet));
        GDX_TRY(check_config(*config));
        int device;
        GDX_TRY(resolve_device(config->device, &device));
        DeviceGuard guard(device);
    
        ConcatText ct;
        uint64_t bad = 0;
        gdx_status st = concat_texts(texts, text_offsets, num_texts, *alphabet, ct, &bad);
        if (st != GDX_OK) {
            t_error_query = bad;
            return fail(st, "text %llu contains a symbol that is not in the alphabet (alphabet.rs:195-198)",
                        (unsigned long long)bad);
        }
        const uint64_t n = ct.text.size();
        if (n > storage_max(config->storage))
            return fail(GDX_ERR_TEXT_TOO_LONG, "text length %llu exceeds the index storage type (construction/mod.rs:34)",
                        (unsigned long long)n);
    
        ImageSources src;
        src.alphabet = alphabet;
        src.storage = config->storage;
        src.sampling_rate = config->suffix_array_sampling_rate;
        src.lookup_depth = config->lookup_table_depth;
        src.n = n;
        src.count = ct.count.data();
        src.sentinels = ct.sentinels.data();
        src.ntexts = num_texts;
        src.accel_flags = accel_flags_from_config(config->flags);
        src.accel_budget = config->accelerator_budget_bytes;
    
        // the dense text goes to the device once: input of the device suffix sort and source of the
        // optional text section of the image
        const bool keep_text = (config->flags & GDX_FLAG_NO_TEXT) == 0;
        const bool keep_isa = keep_text && (config->flags & GDX_FLAG_NO_INVERSE_SAMPLES) == 0;
        uint32_t construction = config->construction;
        if (construction == GDX_CONSTRUCT_AUTO) {  // device suffix sort when the text and its scratch fit
            size_t free_b = 0, total_b = 0;
            construction = GDX_CONSTRUCT_HOST;
            if (n < 0xffffffffull && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && free_b > 36 * n + (1ull << 30))
                construction = GDX_CONSTRUCT_DEVICE;
        }
        ImageHeader h;
        DevMem image;
        {
            DevMem d_text;
            if (keep_text || construction == GDX_CONSTRUCT_DEVICE) {
                CUDA_TRY(d_text.alloc(n));
                CUDA_TRY(cudaMemcpy(d_text.p, ct.text.data(), n, cudaMemcpyHostToDevice));
                if (keep_text) src.d_text = d_text.as<uint8_t>();
            }
            if (construction == GDX_CONSTRUCT_DEVICE) {
                DeviceBuildResult r;
                const bool verify = (config->flags & GDX_FLAG_VERIFY_SUFFIX_ARRAY) != 0;
                const uint32_t rate = config->suffix_array_sampling_rate;
                GDX_TRY(device_build_from_text(nullptr, d_text.as<uint8_t>(), n, alphabet->num_dense_symbols, rate, r,
                                               t_error, false, verify, keep_isa));
                if (verify && r.verify_violations)
                    return fail(GDX_ERR_CUDA, "device suffix array failed verification (%llu violations)",
                                (unsigned long long)r.verify_violations);
                src.border_rows = r.border_rows.data();
                src.border_pos = r.border_pos.data();
                src.n_border = r.border_rows.size();
                src.d_bwt = r.d_bwt.as<uint8_t>();
                src.samples.d = r.d_samples.p;
                src.isa.d = r.d_isa_samples.p;
                GDX_TRY(build_image(src, h, image));
            } else {
                HostParts hp;
                host_parts_from_text(ct.text.data(), n, alphabet->num_dense_symbols,
                                     config->suffix_array_sampling_rate, hp);
                DevMem d_bwt;
                GDX_TRY(upload_bwt(hp.bwt.data(), n, d_bwt));
                src.border_rows = hp.border_rows.data();
                src.border_pos = hp.border_pos.data();
                src.n_border = hp.border_rows.size();
                src.d_bwt = d_bwt.as<uint8_t>();
                src.samples.h64 = hp.samples.data();
                if (keep_isa) src.isa.h64 = hp.isa_samples.data();
                GDX_TRY(build_image(src, h, image));
            }
        }
        return open_index(h, image, device, out);
    });
}

static gdx_status sources_from_parts(const gdx_parts *parts, ImageSources &src,
                                     std::vector<uint64_t> &rows, std::vector<uint64_t> &pos) {
    if (!parts) return fail(GDX_ERR_BAD_ARG, "parts is NULL");
    GDX_TRY(validate_alphabet(parts->alphabet));
    if (parts->sampling_rate == 0) return fail(GDX_ERR_BAD_ARG, "sampling rate must be > 0");
    if (!parts->count || !parts->sentinel_indices || parts->num_texts == 0)
        return fail(GDX_ERR_BAD_ARG, "count / sentinel_indices missing");
    if (parts->text_len > storage_max(parts->storage)) return fail(GDX_ERR_TEXT_TOO_LONG, "text too long for storage");
    // sort the border map by row (it is a HashMap in the reference)
    std::vector<std::pair<uint64_t, uint64_t>> b(parts->num_text_borders);
    for (uint64_t i = 0; i < parts->num_text_borders; ++i)
        b[i] = {parts->text_border_rows[i], parts->text_border_positions[i]};
    std::sort(b.begin(), b.end());
    rows.resize(b.size());
    pos.resize(b.size());
    for (size_t i = 0; i < b.size(); ++i) {
        rows[i] = b[i].first;
        pos[i] = b[i].second;
    }
    src.alphabet = &parts->alphabet;
    src.storage = parts->storage;
    src.sampling_rate = parts->sampling_rate;
    src.lookup_depth = parts->lookup_table_depth;
    src.n = parts->text_len;
    src.count = parts->count;
    src.sentinels = parts->sentinel_indices;
    src.ntexts = parts->num_texts;
    src.border_rows = rows.data();
    src.border_pos = pos.data();
    src.n_border = rows.size();
    if ((parts->sampled_suffix_array != nullptr) == (parts->sampled_suffix_array_u32 != nullptr) && parts->text_len)
        return fail(GDX_ERR_BAD_ARG, "exactly one of sampled_suffix_array / sampled_suffix_array_u32 must be set");
    src.samples.h64 = parts->sampled_suffix_array;
    src.samples.h32 = parts->sampled_suffix_array_u32;
    src.accel_flags = accel_flags_from_config(parts->flags);
    src.accel_budget = parts->accelerator_budget_bytes;
    return GDX_OK;
}

extern "C" gdx_status gdx_index_create_from_bwt(const uint8_t *bwt, const gdx_parts *parts, int32_t device_req,
                                                gdx_index **out) {
    return guarded([&]() -> gdx_status {
        if (!out) return fail(GDX_ERR_BAD_ARG, "out is NULL");
        *out = nullptr;
        if (!bwt) return fail(GDX_ERR_BAD_ARG, "bwt is NULL");
        ImageSources src;
        std::vector<uint64_t> rows, pos;
        GDX_TRY(sources_from_parts(parts, src, rows, pos));
        int device;
        GDX_TRY(resolve_device(device_req, &device));
        DeviceGuard guard(device);
        ImageHeader h;
        DevMem image;
        {
            DevMem d_bwt;
            GDX_TRY(upload_bwt(bwt, src.n, d_bwt));
            src.d_bwt = d_bwt.as<uint8_t>();
            GDX_TRY(build_image(src, h, image));
        }
        return open_index(h, image, device, out);
    });
}

extern "C" gdx_status gdx_index_create_from_parts(const gdx_parts *parts, int32_t device_req, gdx_index **out) {
    return guarded([&]() -> gdx_status {
        if (!out) return fail(GDX_ERR_BAD_ARG, "out is NULL");
        *out = nullptr;
        ImageSources src;
        std::vector<uint64_t> rows, pos;
        GDX_TRY(sources_from_parts(parts, src, rows, pos));
        if (!parts->interleaved_blocks) return fail(GDX_ERR_BAD_ARG, "interleaved_blocks is NULL");
        int device;
        GDX_TRY(resolve_device(device_req, &device));
        DeviceGuard guard(device);
        // the reference's blocks -> dense BWT on the device (symbol_at of the variant), then the common path
        const uint32_t block_bits = parts->block_bits ? parts->block_bits : 64;
        if ((block_bits != 64 && block_bits != 512) || parts->rank_variant > GDX_RANK_FLAT)
            return fail(GDX_ERR_BAD_ARG, "rank_variant must be GDX_RANK_CONDENSED or GDX_RANK_FLAT, block_bits 64 or 512");
        const bool flat = parts->rank_variant == GDX_RANK_FLAT;
        const uint32_t words = block_bits / 64, used = block_bits - (flat ? 16 : 0);
        const uint32_t units = flat ? parts->alphabet.num_dense_symbols : choose_layout(parts->alphabet.num_dense_symbols).planes;
        const uint64_t nwords = div_up(src.n + 1, used) * units * words;
        ImageHeader h;
        DevMem image;
        {
            DevMem d_bwt;
            {
                DevMem d_blocks;
                CUDA_TRY(d_blocks.alloc(nwords * 8));
                cudaError_t e = d_bwt.alloc(src.n);
                if (e == cudaSuccess)
                    e = cudaMemcpy(d_blocks.p, parts->interleaved_blocks, nwords * 8, cudaMemcpyHostToDevice);
                if (e == cudaSuccess && src.n) {
                    k_ref_blocks_to_bwt<<<(unsigned)div_up(src.n, 256), 256>>>(
                        d_blocks.as<uint64_t>(), flat ? 1u : 0u, words, units, src.n, d_bwt.as<uint8_t>());
                    e = cudaGetLastError();
                }
                if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "block upload failed: %s", cudaGetErrorString(e));
            }
            src.d_bwt = d_bwt.as<uint8_t>();
            GDX_TRY(build_image(src, h, image));
        }
        return open_index(h, image, device, out);
    });
}

extern "C" gdx_status gdx_concat_texts(const uint8_t *texts, const uint64_t *text_offsets, uint64_t num_texts,
                                       const gdx_alphabet *alphabet, uint8_t *dense_out, uint64_t *sentinels_out,
                                       uint64_t *count_out) {
    return guarded([&]() -> gdx_status {
        if (!text_offsets || !alphabet || !dense_out || !sentinels_out || !count_out || num_texts == 0)
            return fail(GDX_ERR_BAD_ARG, "NULL argument or no texts");
        GDX_TRY(check_text_offsets(text_offsets, num_texts));
        GDX_TRY(validate_alphabet(*alphabet));
        ConcatText ct;
        uint64_t bad = 0;
        gdx_status st = concat_texts(texts, text_offsets, num_texts, *alphabet, ct, &bad);
        if (st != GDX_OK) {
            t_error_query = bad;
            return fail(st, "text %llu contains a symbol that is not in the alphabet (alphabet.rs:195-198)",
                        (unsigned long long)bad);
        }
        memcpy(dense_out, ct.text.data(), ct.text.size());
        memcpy(sentinels_out, ct.sentinels.data(), ct.sentinels.size() * 8);
        memcpy(count_out, ct.count.data(), ct.count.size() * 8);
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_suffix_array(const uint8_t *dense_text, uint64_t n, uint32_t sigma, uint32_t where,
                                       int32_t device_req, uint64_t *sa_out) {
    return guarded([&]() -> gdx_status {
        if (n == 0) return GDX_OK;
        if (!dense_text || !sa_out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        if (sigma < 2 || sigma > 256) return fail(GDX_ERR_BAD_ARG, "alphabet size must be in [2,256]");
        for (uint64_t i = 0; i < n; ++i)
            if (dense_text[i] >= sigma) return fail(GDX_ERR_BAD_ARG, "symbol %u at %llu is not dense", dense_text[i], (unsigned long long)i);
        if (where == GDX_CONSTRUCT_HOST) {
            std::vector<int64_t> sa;
            suffix_array_sais(dense_text, n, sigma, sa);
            for (uint64_t i = 0; i < n; ++i) sa_out[i] = (uint64_t)sa[i];
            return GDX_OK;
        }
        int device;
        GDX_TRY(resolve_device(device_req, &device));
        DeviceGuard guard(device);
        DeviceBuildResult r;
        gdx_status st = device_build_from_text(dense_text, nullptr, n, sigma, 1, r, t_error, true, true);
        if (st != GDX_OK) return st;
        std::vector<uint32_t> sa32(n);
        cudaError_t e = cudaMemcpy(sa32.data(), r.d_sa.p, n * 4, cudaMemcpyDeviceToHost);
        const uint64_t viol = r.verify_violations;
        r = DeviceBuildResult();
        if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "suffix array download failed: %s", cudaGetErrorString(e));
        for (uint64_t i = 0; i < n; ++i) sa_out[i] = sa32[i];
        if (viol) return fail(GDX_ERR_CUDA, "device suffix array failed verification (%llu violations)", (unsigned long long)viol);
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_download_bwt(const gdx_index *idx, uint8_t *bwt_out) {
    return guarded([&]() -> gdx_status {
        if (!idx || !bwt_out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        DeviceGuard guard(idx->device);
        const uint64_t n = idx->h.n, chunk = 256ull << 20;
        DevMem d;
        CUDA_TRY(d.alloc(std::min<uint64_t>(n, chunk)));
        for (uint64_t b = 0; b < n; b += chunk) {
            const uint64_t e = std::min<uint64_t>(n, b + chunk);
            GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
                k_records_to_bwt<decltype(L)><<<(unsigned)div_up(e - b, 256), 256>>>(idx->dev, b, e, d.as<uint8_t>());
                return GDX_OK;
            }));
            const cudaError_t ce = cudaMemcpy(bwt_out + b, d.p, e - b, cudaMemcpyDeviceToHost);
            if (ce != cudaSuccess) return fail(GDX_ERR_CUDA, "BWT download failed: %s", cudaGetErrorString(ce));
        }
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_download_samples(const gdx_index *idx, uint64_t *samples_out) {
    return guarded([&]() -> gdx_status {
        if (!idx || !samples_out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        DeviceGuard guard(idx->device);
        const uint64_t ns = idx->h.n_samples;
        const uint8_t *src = (const uint8_t *)idx->image + idx->h.off_samples;
        if (idx->h.wide) {
            CUDA_TRY(cudaMemcpy(samples_out, src, ns * 8, cudaMemcpyDeviceToHost));
        } else {
            // narrow samples land in the upper half of the output buffer and are widened in place
            uint32_t *tmp = reinterpret_cast<uint32_t *>(samples_out) + ns;
            CUDA_TRY(cudaMemcpy(tmp, src, ns * 4, cudaMemcpyDeviceToHost));
            for (uint64_t i = 0; i < ns; ++i) samples_out[i] = tmp[i];
        }
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_download_text_borders(const gdx_index *idx, uint64_t *rows_out, uint64_t *positions_out) {
    if (!idx || !rows_out || !positions_out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
    DeviceGuard guard(idx->device);
    const uint8_t *base = (const uint8_t *)idx->image;
    CUDA_TRY(cudaMemcpy(rows_out, base + idx->h.off_border_rows, idx->h.n_border * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(positions_out, base + idx->h.off_border_pos, idx->h.n_border * 8, cudaMemcpyDeviceToHost));
    return GDX_OK;
}

extern "C" gdx_status gdx_index_get_count(const gdx_index *idx, uint64_t *count_out) {
    if (!idx || !count_out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
    DeviceGuard guard(idx->device);
    CUDA_TRY(cudaMemcpy(count_out, (const uint8_t *)idx->image + idx->h.off_count, (uint64_t)(idx->h.sigma + 1) * 8,
                        cudaMemcpyDeviceToHost));
    return GDX_OK;
}

extern "C" void gdx_index_destroy(gdx_index *idx) {
    if (!idx) return;
    DeviceGuard guard(idx->device);
    delete idx;
}

extern "C" gdx_status gdx_index_get_info(const gdx_index *idx, gdx_index_info *out) {
    if (!idx || !out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
    const ImageHeader &h = idx->h;
    out->text_len = h.n;
    out->num_texts = h.ntexts;
    out->num_dense_symbols = h.sigma;
    out->num_searchable_dense_symbols = h.ns;
    out->storage = h.storage;
    out->sampling_rate = h.sampling_rate;
    out->lookup_table_depth = h.lookup_depth;
    out->rank_layout = h.layout.kind;
    out->rank_record_bytes = h.layout.stride;
    out->rank_positions_per_record = 1u << h.layout.log2_pos;
    out->device = idx->device;
    out->image_bytes = h.image_bytes;
    out->rank_bytes = h.off_samples - h.off_records;
    out->sample_bytes = h.off_lookup - h.off_samples;
    out->lookup_bytes = h.off_border_rows - h.off_lookup;
    out->num_samples = h.n_samples;
    out->num_text_borders = h.n_border;
    out->text_bytes = h.text_bits ? h.off_isa - h.off_text : 0;
    out->inverse_sample_bytes = h.has_isa ? h.image_bytes - h.off_isa : 0;
    out->dense_suffix_array_bytes = idx->dense_sa.bytes;
    out->seed_table_bytes = idx->seed_table.bytes;
    out->seed_table_depth = idx->seed_table ? idx->seed_depth : 0;
    out->row_context_entry_bytes = idx->row_context ? 16 : 0;
    out->compact_seed_depth = idx->compact_seed ? idx->compact_depth : 0;
    out->compact_seed_bytes = idx->compact_seed.bytes;
    return GDX_OK;
}

// ================================================================================================
// index files
// ================================================================================================
namespace {
constexpr char kFileMagic[8] = {'G', 'D', 'X', 'F', 'I', 'L', 'E', '1'};
struct FilePrefix {
    char magic[8];
    uint64_t header_bytes, image_bytes, user_bytes;
};
struct FileCloser {
    FILE *f;
    ~FileCloser() {
        if (f) fclose(f);
    }
};
}  // namespace

extern "C" gdx_status gdx_index_save_to_file(const gdx_index *idx, const char *path, const void *user_data,
                                             uint64_t user_bytes) {
    return guarded([&]() -> gdx_status {
        if (!idx || !path || (user_bytes && !user_data)) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        DeviceGuard guard(idx->device);
        FileCloser fc{fopen(path, "wb")};
        if (!fc.f) return fail(GDX_ERR_BAD_ARG, "cannot open %s for writing", path);
        FilePrefix p;
        memcpy(p.magic, kFileMagic, 8);
        p.header_bytes = sizeof(ImageHeader);
        p.image_bytes = idx->h.image_bytes;
        p.user_bytes = user_bytes;
        if (fwrite(&p, sizeof p, 1, fc.f) != 1 || fwrite(&idx->h, sizeof(ImageHeader), 1, fc.f) != 1 ||
            (user_bytes && fwrite(user_data, user_bytes, 1, fc.f) != 1))
            return fail(GDX_ERR_BAD_ARG, "write to %s failed", path);
        const uint64_t chunk = 64ull << 20;
        HBuf stage;
        CUDA_TRY(stage.alloc(chunk));
        for (uint64_t off = 0; off < p.image_bytes; off += chunk) {
            const uint64_t nb = std::min<uint64_t>(chunk, p.image_bytes - off);
            const cudaError_t e = cudaMemcpy(stage.p, (const uint8_t *)idx->image + off, nb, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "image download failed: %s", cudaGetErrorString(e));
            if (fwrite(stage.p, nb, 1, fc.f) != 1) return fail(GDX_ERR_BAD_ARG, "write to %s failed", path);
        }
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_load_from_file(const char *path, int32_t device_req, gdx_index **out,
                                               void *user_data_out, uint64_t user_capacity, uint64_t *user_bytes_out) {
    return guarded([&]() -> gdx_status {
        if (!path || !out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        *out = nullptr;
        FileCloser fc{fopen(path, "rb")};
        if (!fc.f) return fail(GDX_ERR_BAD_ARG, "cannot open %s", path);
        FilePrefix p;
        ImageHeader h;
        if (fread(&p, sizeof p, 1, fc.f) != 1 || memcmp(p.magic, kFileMagic, 8) != 0 || p.header_bytes != sizeof(ImageHeader) ||
            fread(&h, sizeof h, 1, fc.f) != 1 || h.magic != kImageMagic || h.version != GDX_ABI_VERSION ||
            h.image_bytes != p.image_bytes)
            return fail(GDX_ERR_BAD_ARG, "%s is not a genedex_b200 index file of this version", path);
        GDX_TRY(validate_header(h));
        // the sizes in the prefix must add up to the size of the file before anything is allocated from them
        const off_t here = ftello(fc.f);
        if (here < 0 || fseeko(fc.f, 0, SEEK_END) != 0) return fail(GDX_ERR_BAD_ARG, "cannot seek in %s", path);
        const off_t file_size = ftello(fc.f);
        if (fseeko(fc.f, here, SEEK_SET) != 0 || file_size < here || p.user_bytes > (uint64_t)(file_size - here) ||
            p.image_bytes != (uint64_t)(file_size - here) - p.user_bytes)
            return fail(GDX_ERR_BAD_ARG, "%s is truncated or corrupt (section sizes do not add up to the file size)", path);
        if (user_bytes_out) *user_bytes_out = p.user_bytes;
        if (p.user_bytes) {
            const uint64_t keep = user_data_out ? std::min<uint64_t>(p.user_bytes, user_capacity) : 0;
            if (keep && fread(user_data_out, keep, 1, fc.f) != 1) return fail(GDX_ERR_BAD_ARG, "%s is truncated", path);
            if (fseeko(fc.f, here + (off_t)p.user_bytes, SEEK_SET) != 0) return fail(GDX_ERR_BAD_ARG, "cannot seek in %s", path);
        }
        int device;
        GDX_TRY(resolve_device(device_req, &device));
        DeviceGuard guard(device);
        DevMem image;
        CUDA_TRY(image.alloc(p.image_bytes));
        const uint64_t chunk = 64ull << 20;
        HBuf stage;
        if (stage.alloc(chunk) != cudaSuccess) return fail(GDX_ERR_OOM, "pinned staging allocation failed");
        for (uint64_t off = 0; off < p.image_bytes; off += chunk) {
            const uint64_t nb = std::min<uint64_t>(chunk, p.image_bytes - off);
            if (fread(stage.p, nb, 1, fc.f) != 1) return fail(GDX_ERR_BAD_ARG, "%s is truncated", path);
            const cudaError_t e = cudaMemcpy(image.as<uint8_t>() + off, stage.p, nb, cudaMemcpyHostToDevice);
            if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "image upload failed: %s", cudaGetErrorString(e));
        }
        stage.reset();
        return open_index(h, image, device, out);
    });
}

// ================================================================================================
// replication
// ================================================================================================
extern "C" uint64_t gdx_index_header_bytes(void) { return sizeof(ImageHeader); }

extern "C" gdx_status gdx_index_export(const gdx_index *idx, void *header_out, const void **device_image,
                                       uint64_t *image_bytes) {
    if (!idx) return fail(GDX_ERR_BAD_ARG, "idx is NULL");
    if (header_out) memcpy(header_out, &idx->h, sizeof(ImageHeader));
    if (device_image) *device_image = idx->image;
    if (image_bytes) *image_bytes = idx->h.image_bytes;
    return GDX_OK;
}

extern "C" gdx_status gdx_index_adopt_image(const void *header, void *device_image, int32_t device_req,
                                            int32_t own_image, gdx_index **out) {
    return guarded([&]() -> gdx_status {
        if (!header || !device_image || !out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        *out = nullptr;
        ImageHeader h;
        memcpy(&h, header, sizeof h);
        GDX_TRY(validate_header(h));
        int device;
        GDX_TRY(resolve_device(device_req, &device));
        DeviceGuard guard(device);
        return open_index(h, device_image, own_image != 0, device, out);
    });
}

extern "C" gdx_status gdx_index_set_seed_table_depth(gdx_index *idx, int32_t depth) {
    const char *busy = "queries are running on this index: the seed table cannot change now";
    return with_config(idx, busy, [&]() -> gdx_status {
        if (depth > 0) {
            GDX_TRY(build_seed_table(idx, (uint32_t)depth));
            return build_compact_seed(idx);
        }
        drop_table(idx, idx->compact_seed);
        drop_table(idx, idx->seed_table);
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_set_row_context_table(gdx_index *idx, int32_t on) {
    const char *busy = "queries are running on this index: the row context table cannot change now";
    return with_config(idx, busy, [&]() -> gdx_status {
        if (on) return build_row_context(idx);
        drop_table(idx, idx->row_context);
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_set_text_verification(gdx_index *idx, int32_t on) {
    return with_config(idx, "queries are running on this index", [&]() -> gdx_status {
        idx->verify = on != 0;
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_index_set_dense_suffix_array(gdx_index *idx, int32_t on) {
    const char *busy = "queries are running on this index: the dense suffix array cannot change now";
    return with_config(idx, busy, [&]() -> gdx_status {
        if (on) return build_dense_sa(idx);
        drop_table(idx, idx->dense_sa);
        return GDX_OK;
    });
}

// ---- NCCL, loaded at run time ---------------------------------------------------------------------------
// The library does not link libnccl: a process that already carries one (PyTorch bundles its own libnccl.so.2)
// must not get a second copy, and single-GPU users need none.  The handful of entry points used here has been
// ABI-stable since NCCL 2.
namespace {
struct Nccl {
    typedef struct ncclComm *comm_t;
    struct unique_id {
        char internal[GDX_NCCL_UNIQUE_ID_BYTES];
    };
    int (*GetUniqueId)(unique_id *) = nullptr;
    int (*CommInitRank)(comm_t *, int, unique_id, int) = nullptr;
    int (*CommInitAll)(comm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(comm_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int /*ncclDataType_t*/, int, comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
    std::string why;
    static constexpr int kUint8 = 1;  // ncclUint8
};

const Nccl &nccl() {
    static const Nccl n = [] {
        Nccl r;
        const char *names[] = {getenv("GDX_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        void *h = nullptr;
        for (const char *nm : names)
            if (nm && *nm && (h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break;
        if (!h) {
            r.why = "libnccl.so.2 could not be loaded";
            return r;
        }
        auto sym = [&](const char *name) { return dlsym(h, name); };
        r.GetUniqueId = (decltype(r.GetUniqueId))sym("ncclGetUniqueId");
        r.CommInitRank = (decltype(r.CommInitRank))sym("ncclCommInitRank");
        r.CommInitAll = (decltype(r.CommInitAll))sym("ncclCommInitAll");
        r.CommDestroy = (decltype(r.CommDestroy))sym("ncclCommDestroy");
        r.Broadcast = (decltype(r.Broadcast))sym("ncclBroadcast");
        r.GroupStart = (decltype(r.GroupStart))sym("ncclGroupStart");
        r.GroupEnd = (decltype(r.GroupEnd))sym("ncclGroupEnd");
        r.GetErrorString = (decltype(r.GetErrorString))sym("ncclGetErrorString");
        r.ok = r.GetUniqueId && r.CommInitRank && r.CommInitAll && r.CommDestroy && r.Broadcast && r.GroupStart &&
               r.GroupEnd && r.GetErrorString;
        if (!r.ok) r.why = "libnccl.so.2 lacks an expected entry point";
        return r;
    }();
    return n;
}

#define NCCL_TRY(expr)                                                                                     \
    do {                                                                                                   \
        int _r = (expr);                                                                                   \
        if (_r != 0) return fail(GDX_ERR_CUDA, "%s failed: %s", #expr, nccl().GetErrorString(_r));         \
    } while (0)

thread_local const char *t_transport = "";
constexpr uint64_t kBroadcastPiece = 1ull << 30;
}  // namespace

extern "C" const char *gdx_replicate_transport(void) { return t_transport; }

extern "C" gdx_status gdx_index_replicate(const gdx_index *idx, const int32_t *devices, int32_t n_devices,
                                          gdx_index **out_replicas) {
    return guarded([&]() -> gdx_status {
        if (!idx || !devices || !out_replicas || n_devices < 0) return fail(GDX_ERR_BAD_ARG, "bad argument");
        t_transport = "";
        for (int i = 0; i < n_devices; ++i) out_replicas[i] = nullptr;
        std::vector<int> dev(n_devices);
        for (int i = 0; i < n_devices; ++i) GDX_TRY(resolve_device(devices[i], &dev[i]));
        // the images not yet opened as replicas, each freed with its device current
        struct Images {
            const std::vector<int> &dev;
            std::vector<DevMem> img;
            ~Images() {
                for (size_t i = 0; i < img.size(); ++i)
                    if (img[i]) {
                        DeviceGuard g(dev[i]);
                        img[i].reset();
                    }
            }
        } images{dev, std::vector<DevMem>(n_devices)};
        std::vector<DevMem> &img = images.img;
        const uint64_t bytes = idx->h.image_bytes;
        for (int i = 0; i < n_devices; ++i) {
            DeviceGuard g(dev[i]);
            const cudaError_t e = img[i].alloc(bytes);
            if (e != cudaSuccess) return fail(GDX_ERR_OOM, "replica on device %d: %s", dev[i], cudaGetErrorString(e));
        }
        // communicator over the source device + every distinct other target; targets on the source device (and
        // repeated targets) are filled by device-to-device copies afterwards
        std::vector<int> comm_dev{idx->device};
        std::vector<int> member(n_devices, -1);  // rank of target i in the communicator, -1 = copy
        for (int i = 0; i < n_devices; ++i) {
            if (std::find(comm_dev.begin(), comm_dev.end(), dev[i]) != comm_dev.end()) continue;
            member[i] = (int)comm_dev.size();
            comm_dev.push_back(dev[i]);
        }
        const bool want_nccl = comm_dev.size() > 1 && !(getenv("GDX_REPLICATE") && strcmp(getenv("GDX_REPLICATE"), "peer") == 0);
        bool done = comm_dev.size() <= 1;
        if (want_nccl && nccl().ok) {
            const Nccl &N = nccl();
            const int world = (int)comm_dev.size();
            std::vector<Nccl::comm_t> comms(world, nullptr);
            std::vector<Stream> streams(world);
            gdx_status st = [&]() -> gdx_status {
                NCCL_TRY(N.CommInitAll(comms.data(), world, comm_dev.data()));
                for (int r = 0; r < world; ++r) {
                    DeviceGuard g(comm_dev[r]);
                    CUDA_TRY(streams[r].create(cudaStreamNonBlocking));
                }
                for (uint64_t off = 0; off < bytes; off += kBroadcastPiece) {
                    const uint64_t nb = std::min(kBroadcastPiece, bytes - off);
                    NCCL_TRY(N.GroupStart());
                    for (int r = 0; r < world; ++r) {
                        void *recv = (uint8_t *)idx->image + off;  // root: in place
                        for (int i = 0; i < n_devices && r > 0; ++i)
                            if (member[i] == r) recv = img[i].as<uint8_t>() + off;
                        DeviceGuard g(comm_dev[r]);
                        NCCL_TRY(N.Broadcast((const uint8_t *)idx->image + off, recv, nb, Nccl::kUint8, 0, comms[r], streams[r]));
                    }
                    NCCL_TRY(N.GroupEnd());
                }
                for (int r = 0; r < world; ++r) {
                    DeviceGuard g(comm_dev[r]);
                    CUDA_TRY(cudaStreamSynchronize(streams[r]));
                }
                return GDX_OK;
            }();
            for (int r = 0; r < world; ++r) {
                DeviceGuard g(comm_dev[r]);
                streams[r] = Stream();
                if (comms[r]) N.CommDestroy(comms[r]);
            }
            if (st != GDX_OK) return st;
            t_transport = "nccl";
            done = true;
        }
        for (int i = 0; i < n_devices; ++i) {
            if (done && member[i] >= 0) continue;
            // same device as the source or as an earlier target (or no NCCL): a plain copy
            DeviceGuard g(dev[i]);
            const void *from = idx->image;
            int from_dev = idx->device;
            if (done && member[i] < 0 && dev[i] != idx->device)
                for (int j = 0; j < i; ++j)
                    if (dev[j] == dev[i] && member[j] >= 0) {
                        from = img[j].p;
                        from_dev = dev[j];
                    }
            const cudaError_t e = cudaMemcpyPeer(img[i].p, dev[i], from, from_dev, bytes);
            if (e != cudaSuccess) return fail(GDX_ERR_CUDA, "copy to device %d failed: %s", dev[i], cudaGetErrorString(e));
            if (!done && *t_transport == 0) t_transport = "peer";
        }
        if (*t_transport == 0) t_transport = "peer";
        for (int i = 0; i < n_devices; ++i) {
            DeviceGuard g(dev[i]);
            const gdx_status st = open_index(idx->h, img[i], dev[i], &out_replicas[i]);
            if (st != GDX_OK) {
                for (int j = 0; j < i; ++j) {
                    gdx_index_destroy(out_replicas[j]);
                    out_replicas[j] = nullptr;
                }
                return st;
            }
        }
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_nccl_unique_id(void *id_out) {
    if (!id_out) return fail(GDX_ERR_BAD_ARG, "id_out is NULL");
    if (!nccl().ok) return fail(GDX_ERR_UNSUPPORTED, "NCCL is not available: %s", nccl().why.c_str());
    Nccl::unique_id id;
    NCCL_TRY(nccl().GetUniqueId(&id));
    memcpy(id_out, &id, sizeof id);
    return GDX_OK;
}

extern "C" gdx_status gdx_index_broadcast(const gdx_index *src, const void *unique_id, int32_t rank, int32_t world,
                                          int32_t root, int32_t device_req, gdx_index **out) {
    return guarded([&]() -> gdx_status {
        if (!out || !unique_id || world < 1 || rank < 0 || rank >= world || root < 0 || root >= world)
            return fail(GDX_ERR_BAD_ARG, "bad argument");
        *out = nullptr;
        if ((rank == root) != (src != nullptr)) return fail(GDX_ERR_BAD_ARG, "src must be given on the root rank and only there");
        if (!nccl().ok) return fail(GDX_ERR_UNSUPPORTED, "NCCL is not available: %s", nccl().why.c_str());
        const Nccl &N = nccl();
        int device;
        GDX_TRY(resolve_device(rank == root ? src->device : device_req, &device));
        DeviceGuard guard(device);
        Nccl::unique_id id;
        memcpy(&id, unique_id, sizeof id);
        Nccl::comm_t comm = nullptr;
        NCCL_TRY(N.CommInitRank(&comm, world, id, rank));
        DevMem image;  // of a receiving rank
        ImageHeader h;
        const gdx_status st = [&]() -> gdx_status {
            Stream stream;
            DevMem d_hdr;
            CUDA_TRY(stream.create(cudaStreamNonBlocking));
            CUDA_TRY(d_hdr.alloc(sizeof(ImageHeader)));
            if (rank == root) CUDA_TRY(cudaMemcpyAsync(d_hdr.p, &src->h, sizeof(ImageHeader), cudaMemcpyHostToDevice, stream));
            NCCL_TRY(N.Broadcast(d_hdr.p, d_hdr.p, sizeof(ImageHeader), Nccl::kUint8, root, comm, stream));
            CUDA_TRY(cudaMemcpyAsync(&h, d_hdr.p, sizeof(ImageHeader), cudaMemcpyDeviceToHost, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
            GDX_TRY(validate_header(h));
            if (rank != root) CUDA_TRY(image.alloc(h.image_bytes));
            uint8_t *img = rank == root ? (uint8_t *)src->image : image.as<uint8_t>();
            for (uint64_t off = 0; off < h.image_bytes; off += kBroadcastPiece) {
                const uint64_t nb = std::min(kBroadcastPiece, h.image_bytes - off);
                NCCL_TRY(N.Broadcast(img + off, img + off, nb, Nccl::kUint8, root, comm, stream));
            }
            CUDA_TRY(cudaStreamSynchronize(stream));
            return GDX_OK;
        }();
        N.CommDestroy(comm);
        if (st != GDX_OK) return st;
        t_transport = "nccl";
        if (rank == root) {
            *out = const_cast<gdx_index *>(src);
            return GDX_OK;
        }
        return open_index(h, image, device, out);
    });
}

// ================================================================================================
// search
// ================================================================================================
namespace {

bool verify_enabled() {
    static const bool on = [] {
        const char *e = getenv("GDX_VERIFY");
        return !e || atoi(e) != 0;
    }();
    return on;
}

// mode 0: cursors (starts, ends); 1: counts; 2: locate intervals (interval or resolved hit);
// narrow: results are written as uint32 (modes 0 and 1, texts shorter than 2^32)
template <class L>
void launch_search(const gdx_index *idx, const DevQueries &dq, uint64_t *a, uint64_t *b, int mode, bool narrow,
                   uint64_t qbase, uint64_t *err, SearchCounters *stats, const uint32_t *perm,
                   const uint32_t *slot_map, cudaStream_t stream) {
    if (dq.nq == 0) return;
    const unsigned grid = (unsigned)div_up(dq.nq, 256);
    const bool verify = idx->dev.text && idx->verify;
    const int mf = mode | (narrow ? kModeNarrow : 0);
#define GDX_LAUNCH(V, C, P) k_search<L, V, C, P><<<grid, 256, 0, stream>>>(idx->dev, dq, a, b, mf, qbase, err, stats, perm, slot_map)
    if (dq.packed) {
        if (verify && mode != 0) GDX_LAUNCH(true, false, true);
        else if (verify && idx->dev.isa) GDX_LAUNCH(true, true, true);
        else GDX_LAUNCH(false, false, true);
    } else {
        if (verify && mode != 0) GDX_LAUNCH(true, false, false);
        else if (verify && idx->dev.isa) GDX_LAUNCH(true, true, false);
        else GDX_LAUNCH(false, false, false);
    }
#undef GDX_LAUNCH
}

// ---- suffix sort of a query batch (locality of the first search steps, see k_query_keys) -------------
constexpr uint64_t kSortMinQueries = 1ull << 15;

bool sort_enabled() {
    static const bool on = [] {
        const char *e = getenv("GDX_SORT_QUERIES");
        return !e || atoi(e) != 0;
    }();
    return on;
}

struct SortPlan {
    uint32_t key_bits = 0, key_syms = 0;
    size_t tmp_bytes = 0;
    uint64_t total_bytes = 0;  // keys a/b + idx a/b + cub temp, 256 B aligned pieces
    bool use = false;
};

// fixed_len: length of every query of the batch, 0 = variable
SortPlan plan_sort(const gdx_index *idx, uint64_t nq, uint64_t fixed_len) {
    SortPlan p;
    if (!sort_enabled() || nq < kSortMinQueries || nq >= 0xffffffffull) return p;
    // The sort makes neighbouring threads share the first ~log_ns(nq) search steps.  When a lookup level
    // (configured, or the seed table accelerator) already replaces that many steps there is nothing left to
    // share: reading the queries in their own order is then cheaper (coalesced, no sort): 1.39 vs 2.01 ms per
    // 7.5 M queries at depth 13.
    {
        uint32_t d = idx->h.lookup_depth;
        if (idx->dev.seed_lookup && idx->dev.seed_depth > d && (fixed_len == 0 || fixed_len >= idx->dev.seed_depth))
            d = idx->dev.seed_depth;
        const uint64_t entries = seed_entries(idx->h.ns, d);
        if (d > 0 && (entries == 0 || entries >= nq)) return p;
    }
    uint32_t bits = 1;
    while ((1u << bits) < idx->h.ns) ++bits;
    p.key_bits = bits;
    p.key_syms = std::min<uint32_t>(32 / bits, 12);  // DNA: 24-bit keys = 3 radix passes, 4^12 > any batch
    cub::DoubleBuffer<uint32_t> dk(nullptr, nullptr), dv(nullptr, nullptr);
    if (cub::DeviceRadixSort::SortPairs(nullptr, p.tmp_bytes, dk, dv, (int64_t)nq, 0, (int)(p.key_bits * p.key_syms)) !=
        cudaSuccess)
        return p;
    p.total_bytes = 4 * align_up(nq * 4, 256) + align_up(p.tmp_bytes, 256);
    p.use = true;
    return p;
}

// scratch: total_bytes of device memory; returns the permutation (sorted query indices) in *perm
gdx_status sort_queries(const gdx_index *idx, const DevQueries &dq, const SortPlan &p, void *scratch,
                        cudaStream_t stream, const uint32_t **perm) {
    uint8_t *base = (uint8_t *)scratch;
    const uint64_t piece = align_up(dq.nq * 4, 256);
    uint32_t *ka = (uint32_t *)base, *kb = (uint32_t *)(base + piece), *ia = (uint32_t *)(base + 2 * piece),
             *ib = (uint32_t *)(base + 3 * piece);
    void *tmp = base + 4 * piece;
    k_query_keys<<<(unsigned)div_up(dq.nq, 256), 256, 0, stream>>>(idx->dev, dq, p.key_bits, p.key_syms, ka, ia);
    CUDA_TRY(cudaGetLastError());
    cub::DoubleBuffer<uint32_t> dk(ka, kb), dv(ia, ib);
    size_t tb = p.tmp_bytes;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(tmp, tb, dk, dv, (int64_t)dq.nq, 0, (int)(p.key_bits * p.key_syms), stream));
    *perm = dv.Current();
    return GDX_OK;
}

gdx_status check_queries(const gdx_index *idx, const gdx_queries *q) {
    if (!q) return fail(GDX_ERR_BAD_ARG, "queries is NULL");
    if (q->offsets && q->nq && q->offsets[q->nq] < q->offsets[0])
        return fail(GDX_ERR_BAD_ARG, "queries->offsets must be non-decreasing");
    if (q->nq && !q->offsets && q->fixed_len && !q->bytes) return fail(GDX_ERR_BAD_ARG, "queries->bytes is NULL");
    if (q->encoding > GDX_QUERIES_PACKED_2BIT) return fail(GDX_ERR_BAD_ARG, "unknown queries->encoding %u", q->encoding);
    if (q->encoding == GDX_QUERIES_PACKED_2BIT && idx && idx->h.ns > 4)
        return fail(GDX_ERR_UNSUPPORTED, "2-bit packed queries need an alphabet with at most 4 searchable symbols (this one has %u)",
                    idx->h.ns);
    return GDX_OK;
}

// index of the first symbol of query i in the batch's symbol stream (IO bytes or 2-bit codes)
uint64_t query_bytes_end(const gdx_queries *q, uint64_t i) {
    return q->offsets ? q->offsets[i] : i * q->fixed_len + q->first_symbol;
}

bool env_flag(const char *name, bool dflt) {
    const char *e = getenv(name);
    return e ? atoi(e) != 0 : dflt;
}
// host-side 2-bit packing of large IO-byte batches (GDX_PACK_QUERIES=0 switches it off for A/B runs)
bool pack_enabled() {
    static const bool on = env_flag("GDX_PACK_QUERIES", true);
    return on;
}
// results of large batches cross PCIe as uint32 when the text is shorter than 2^32 (GDX_NARROW_RESULTS=0: off)
bool narrow_enabled() {
    static const bool on = env_flag("GDX_NARROW_RESULTS", true);
    return on;
}
const uint64_t kPackMinBytes = env_bytes("GDX_PACK_MIN_BYTES", 1ull << 20);

gdx_status acquire_pinned_hits(const gdx_index *idx, uint64_t bytes, void **out, uint64_t *cap_out);
void release_pinned_hits(const gdx_index *idx, void *p);

// a library-owned pinned buffer the results of a call are appended to.  It grows to twice the size asked for (at least
// 4096 bytes) and keeps what it holds; no copy into it may be in flight then.  Unless it is handed over to the caller,
// it goes back to the pool when it dies, which must be after with_workspace drained the streams of a failed call: copies
// into it may still be in flight until then.
struct PinnedResult {
    const gdx_index *idx;
    void *p = nullptr;
    uint64_t cap = 0, used = 0;  // bytes
    explicit PinnedResult(const gdx_index *i) : idx(i) {}
    PinnedResult(const PinnedResult &) = delete;
    PinnedResult &operator=(const PinnedResult &) = delete;
    ~PinnedResult() {
        if (p) release_pinned_hits(idx, p);
    }
    gdx_status reserve(uint64_t bytes) {
        if (bytes <= cap) return GDX_OK;
        void *bigger = nullptr;
        uint64_t c = 0;
        GDX_TRY(acquire_pinned_hits(idx, std::max<uint64_t>(2 * bytes, 4096), &bigger, &c));
        if (p) {
            memcpy(bigger, p, used);
            release_pinned_hits(idx, p);
        }
        p = bigger;
        cap = c;
        return GDX_OK;
    }
    void *hand_over() { return std::exchange(p, nullptr); }
};

// the two-call CUB exclusive scan (size query, then the scan) with its temporary storage in tmp
gdx_status exclusive_sum(DevMem &tmp, uint64_t *in, uint64_t *out, uint64_t n, cudaStream_t st) {
    size_t bytes = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, n, st));
    CUDA_TRY(tmp.reserve(bytes));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(tmp.p, bytes, in, out, n, st));
    return GDX_OK;
}

// K3 + K4 over `n_hits` rows.  With a sampled suffix array (walks of geometric length) the compacting kernel
// keeps every lane busy; with the dense array (one load per row) the plain one-thread-per-hit kernel is the
// shorter program.
template <class L>
void launch_locate_walk(const gdx_index *idx, const uint64_t *rows, uint64_t n_hits, ulonglong2 *hits,
                        unsigned long long *d_walk, cudaStream_t stream, bool hit32 = false) {
    if (idx->dev.sampling_rate > 1)
        k_locate_walk_compact<L><<<(unsigned)div_up(n_hits, kWalkSlice), 256, 0, stream>>>(idx->dev, rows, n_hits, hits, d_walk,
                                                                                           hit32 ? 1 : 0);
    else
        k_locate_walk<L><<<(unsigned)div_up(n_hits, 256), 256, 0, stream>>>(idx->dev, rows, n_hits, hits, d_walk, hit32 ? 1 : 0);
}

// widths -> CSR offsets -> totals to the host (ev_total); does not wait for them
gdx_status IntervalHits::count(cudaStream_t st, const uint64_t *starts, const uint64_t *ends, uint64_t n) {
    CUDA_TRY(counts.reserve((n + 1) * 8));
    CUDA_TRY(offsets.reserve((n + 1) * 8));
    CUDA_TRY(cudaMemsetAsync(d(), 0, sizeof(DeviceWords), st));
    CUDA_TRY(cudaMemsetAsync(counts.as<uint64_t>() + n, 0, 8, st));
    if (n) k_interval_counts<<<(unsigned)div_up(n, 256), 256, 0, st>>>(starts, ends, n, counts.as<uint64_t>(), &d()->wide);
    GDX_TRY(exclusive_sum(scan_tmp, counts.as<uint64_t>(), offsets.as<uint64_t>(), n + 1, st));
    CUDA_TRY(cudaMemcpyAsync(&h()->hits, offsets.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&h()->wide, &d()->wide, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(ev_total, st));
    t_stats.kernel_launches += 2;
    return GDX_OK;
}

// once the totals of count() are known (n_hits > 0): rows of every interval, then the walk to the hits
gdx_status IntervalHits::expand_walk(const gdx_index *idx, cudaStream_t st, const uint64_t *starts, const uint64_t *ends,
                                     uint64_t n, uint64_t n_hits, uint64_t n_wide, unsigned long long *walk_steps,
                                     bool hit32) {
    if (n_hits * 24 > rows.bytes + hits.bytes) {  // 8 B of rows + 16 B of hits per hit
        size_t free_b = 0, total_b = 0;
        CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        if (n_hits * 24 > free_b + rows.bytes + hits.bytes)
            return fail(GDX_ERR_OOM, "%llu hits of one chunk do not fit into device memory; split the batch",
                        (unsigned long long)n_hits);
    }
    CUDA_TRY(rows.reserve(n_hits * 8));
    CUDA_TRY(hits.reserve(n_hits * 16));
    CUDA_TRY(wide.reserve((n_wide + 1) * 8));
    k_expand_rows<<<(unsigned)div_up(n, 256), 256, 0, st>>>(starts, ends, offsets.as<uint64_t>(), n, rows.as<uint64_t>(),
                                                           wide.as<uint64_t>(), &d()->cursor);
    if (n_wide) {
        dim3 grid((unsigned)n_wide, 32);
        k_expand_big_rows<<<grid, 256, 0, st>>>(starts, ends, offsets.as<uint64_t>(), wide.as<uint64_t>(),
                                                rows.as<uint64_t>());
    }
    GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
        launch_locate_walk<decltype(L)>(idx, rows.as<uint64_t>(), n_hits, hits.as<ulonglong2>(), walk_steps, st, hit32);
        return GDX_OK;
    }));
    CUDA_TRY(cudaGetLastError());
    t_stats.kernel_launches += 2 + (n_wide ? 1 : 0);
    return GDX_OK;
}

// host -> device copies on one stream: the bytes they put on the link, and whether one read pinned staging (busy till done)
struct Uploads {
    cudaStream_t st = nullptr;
    uint64_t bytes = 0;
    bool staged = false;
    // through the pinned buffer `stage` (filled by the pool) unless stage is NULL or src already lies in it
    cudaError_t copy(void *dst, const void *src, uint64_t n, HBuf *stage = nullptr) {
        if (stage && src != stage->p) {
            const cudaError_t e = stage->reserve(n);
            if (e != cudaSuccess) return e;
            HostPool::get().copy(stage->p, src, n);
            src = stage->p;
        }
        staged |= stage != nullptr;
        bytes += n;
        return cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, st);
    }
};

// grow device buffers of one stream; growing one frees the old buffer, which is only safe once the stream has drained
gdx_status reserve_drained(cudaStream_t st, std::initializer_list<std::pair<DevMem *, uint64_t>> bufs) {
    if (std::any_of(bufs.begin(), bufs.end(), [](const std::pair<DevMem *, uint64_t> &b) { return b.first->bytes < b.second; }))
        CUDA_TRY(cudaStreamSynchronize(st));
    for (const auto &b : bufs) CUDA_TRY(b.first->reserve(b.second));
    return GDX_OK;
}

gdx_status bad_offsets(uint64_t q) {
    t_error_query = q;
    return fail(GDX_ERR_BAD_ARG, "query %llu: queries->offsets must not decrease and must stay inside the batch",
                (unsigned long long)q);
}

// The error word of k_search / k_hamming: kNoError, or the smallest failing query -- with kBadOffsetFlag when its offsets
// leave the uploaded chunk, else it holds a symbol the kernel refuses (message `invalid`).
gdx_status kernel_error(uint64_t bad, const char *invalid) {
    if (bad == kNoError) return GDX_OK;
    if (bad & kBadOffsetFlag) return bad_offsets(bad & ~kBadOffsetFlag);
    t_error_query = bad;
    return fail(GDX_ERR_INVALID_SYMBOL, "query %llu: %s", (unsigned long long)bad, invalid);
}

// A chunk [q0, q0 + cq) of a slot.  As a handover: its results are on their way into the slot's pinned staging (until
// ev_out), and the sink hands them to the caller one chunk later, while the copy of the next chunk is in flight.
struct Handover {
    Slot *sl = nullptr;
    uint64_t q0 = 0, cq = 0;
    // after the D2H of a chunk into s's staging: mark its end, hand the chunk before over (sink.hand_over)
    template <class Sink>
    gdx_status defer(Slot &s, uint64_t q0_, uint64_t cq_, Sink &sink) {
        CUDA_TRY(cudaEventRecord(s.ev_out, s.stream));
        return std::exchange(*this, Handover{&s, q0_, cq_}).flush(sink);
    }
    template <class Sink>
    gdx_status flush(Sink &sink) {
        Slot *s = std::exchange(sl, nullptr);
        if (!s) return GDX_OK;
        CUDA_TRY(cudaEventSynchronize(s->ev_out));
        sink.hand_over(*s, q0, cq);
        return GDX_OK;
    }
};

// State of a pipelined gdx_locate_many: every chunk of the search pipeline continues, on its own
// stream, with counts -> scan -> expand -> walk -> D2H of its hits, so that the locate kernels and the
// hit copies of chunk k overlap the query upload of the later chunks.
struct LocatePipe {
    static constexpr int mode = 2;  // k_search: interval, or resolved text position for verified queries
    static constexpr bool narrow = false, writes_b = true;
    static constexpr uint32_t stage_elem = 0;
    static constexpr uint64_t d2h = 0;  // (the locate chain counts its copies in t_stats itself)
    const gdx_index *idx;
    Workspace *ws;
    PinnedResult &res;      // the hits of all finished chunks
    uint64_t *hit_offsets;  // caller's array, nq + 1 entries (NULL in the compact form)
    uint32_t *hit_counts = nullptr;  // compact form: hits per query, nq entries, instead of the CSR offsets
    uint64_t hit_bytes = sizeof(gdx_hit);  // 16, or 8 for gdx_hit32
    bool stage_offsets = false;  // the caller's hit_offsets array is pageable
    // chunks whose hit totals are on their way to the host, oldest first.  A chunk is finished two chunks after
    // it was issued (kSlots - 1): by then its total has long arrived, so the issuing thread never waits for a
    // search kernel -- and its slot is only reused by the chunk after that.
    std::deque<Handover> pending;
    Handover staged;  // offsets (or counts) of the last finished chunk
    // widths, exclusive scan, totals to the host; the oldest chunk is finished meanwhile
    gdx_status chunk(Slot &sl, uint64_t q0, uint64_t cq) {
        GDX_TRY(sl.locate.count(sl.stream, sl.out_a.as<uint64_t>(), sl.out_b.as<uint64_t>(), cq));
        pending.push_back(Handover{&sl, q0, cq});
        return pending.size() < (size_t)kSlots ? GDX_OK : finish_oldest();
    }
    gdx_status finish() {
        while (!pending.empty()) GDX_TRY(finish_oldest());
        return staged.flush(*this);
    }
    // per query: global CSR offsets (u64), or in the compact form just the number of hits (u32)
    uint64_t per_q() const { return hit_counts ? 4 : 8; }
    void *dst(uint64_t q0) const { return hit_counts ? (void *)(hit_counts + q0) : (void *)(hit_offsets + q0); }
    void hand_over(Slot &s, uint64_t q0, uint64_t cq) { HostPool::get().copy(dst(q0), s.h_out_a.p, cq * per_q()); }
    // once the chunk's number of hits is known: expand, walk, copy hits + global offsets out
    gdx_status finish_oldest() {
        const Handover p = pending.front();
        pending.pop_front();
        Slot &sl = *p.sl;
        IntervalHits &ih = sl.locate;
        const uint64_t cq = p.cq, q0 = p.q0;
        CUDA_TRY(cudaEventSynchronize(ih.ev_total));
        const uint64_t n_hits = ih.h()->hits, base = res.used / hit_bytes;
        if (n_hits) {
            if ((base + n_hits) * hit_bytes > res.cap) {  // grow the pinned result buffer (rare)
                // the hits of earlier chunks may still be on their way into it, on any slot stream
                for (int s2 = 0; s2 < kSlots; ++s2) CUDA_TRY(cudaStreamSynchronize(ws->slot[s2].stream));
                GDX_TRY(res.reserve((base + n_hits) * hit_bytes));
            }
            const EventPairs::Pair ev = ih.timing.next();
            CUDA_TRY(cudaEventRecord(ev.begin, sl.stream));
            GDX_TRY(ih.expand_walk(idx, sl.stream, sl.out_a.as<uint64_t>(), sl.out_b.as<uint64_t>(), cq, n_hits, ih.h()->wide,
                                   &ws->cnt_d()->locate_walk_steps, hit_bytes == 8));
            CUDA_TRY(cudaEventRecord(ev.end, sl.stream));
            CUDA_TRY(cudaMemcpyAsync((uint8_t *)res.p + res.used, ih.hits.p, n_hits * hit_bytes, cudaMemcpyDeviceToHost,
                                     sl.stream));
            t_stats.d2h_bytes += n_hits * hit_bytes;
        }
        // (compact form: the counts are narrowed into the offsets buffer, which the expansion above no longer needs)
        const uint64_t per_q = this->per_q();
        if (hit_counts) k_narrow_u64<<<(unsigned)div_up(cq, 256), 256, 0, sl.stream>>>(ih.counts.as<uint64_t>(), cq, ih.offsets.as<uint32_t>());
        else k_add_base<<<(unsigned)div_up(cq, 256), 256, 0, sl.stream>>>(ih.offsets.as<uint64_t>(), cq, base);
        CUDA_TRY(cudaGetLastError());
        if (stage_offsets) {
            CUDA_TRY(sl.h_out_a.reserve(cq * per_q));
            CUDA_TRY(cudaMemcpyAsync(sl.h_out_a.p, ih.offsets.p, cq * per_q, cudaMemcpyDeviceToHost, sl.stream));
            GDX_TRY(staged.defer(sl, q0, cq, *this));
        } else {
            CUDA_TRY(cudaMemcpyAsync(dst(q0), ih.offsets.p, cq * per_q, cudaMemcpyDeviceToHost, sl.stream));
        }
        t_stats.d2h_bytes += cq * per_q;
        t_stats.kernel_launches += 1;
        res.used += n_hits * hit_bytes;
        return GDX_OK;
    }
};

// Counts (mode 1) or cursors (mode 0: out_a and out_b) of gdx_count_many / gdx_cursors_many: D2H straight into the
// caller's arrays, or into the slots' pinned staging, handed over by the pool one chunk later.  The results are uint32
// on the device for the u32 entry points and for large batches of the u64 ones (widened on the way out); pinned uint64
// result arrays are filled by DMA without any CPU work, so they stay 64-bit on the wire.
struct CountSink {
    uint8_t *out_a, *out_b;
    uint32_t out_elem;  // bytes per element of the caller's arrays: 8, or 4 for the *_u32 entry points
    int mode;
    bool writes_b, narrow, widen, stage;
    uint32_t dev_elem, stage_elem;  // bytes per result on the device (and on the wire); in staging (0: none)
    uint64_t d2h = 0;  // bytes of the D2H copies
    Handover staged;
    CountSink(const gdx_index *idx, uint64_t nq, void *a, void *b, uint32_t elem, int mode_)
        : out_a((uint8_t *)a), out_b((uint8_t *)b), out_elem(elem), mode(mode_), writes_b(mode_ == 0) {
        const bool large = nq * 8 >= kStageMinBytes;
        narrow = nq && !idx->h.wide &&
                 (out_elem == 4 || (large && narrow_enabled() && !(is_pinned(out_a) && (mode != 0 || is_pinned(out_b)))));
        widen = narrow && out_elem == 8;
        stage = nq && (widen || (large && !is_pinned(out_a)));
        dev_elem = narrow ? 4 : 8;  // (= out_elem unless the results are staged: widening implies staging)
        stage_elem = stage ? dev_elem : 0;
    }
    gdx_status chunk(Slot &sl, uint64_t q0, uint64_t cq) {
        const uint64_t n = cq * dev_elem;
        CUDA_TRY(sl.h_out_a.reserve(cq * stage_elem));
        CUDA_TRY(sl.h_out_b.reserve(writes_b ? cq * stage_elem : 0));
        CUDA_TRY(cudaMemcpyAsync(stage ? sl.h_out_a.p : out_a + q0 * out_elem, sl.out_a.p, n, cudaMemcpyDeviceToHost, sl.stream));
        if (writes_b)
            CUDA_TRY(cudaMemcpyAsync(stage ? sl.h_out_b.p : out_b + q0 * out_elem, sl.out_b.p, n, cudaMemcpyDeviceToHost, sl.stream));
        d2h += n * (writes_b ? 2 : 1);
        return stage ? staged.defer(sl, q0, cq, *this) : GDX_OK;
    }
    gdx_status finish() { return staged.flush(*this); }
    void hand_over(Slot &s, uint64_t q0, uint64_t cq) {
        if (widen) {
            HostPool::get().widen_u32((uint64_t *)out_a + q0, (const uint32_t *)s.h_out_a.p, cq);
            if (writes_b) HostPool::get().widen_u32((uint64_t *)out_b + q0, (const uint32_t *)s.h_out_b.p, cq);
        } else {
            HostPool::get().copy(out_a + q0 * out_elem, s.h_out_a.p, cq * out_elem);
            if (writes_b) HostPool::get().copy(out_b + q0 * out_elem, s.h_out_b.p, cq * out_elem);
        }
    }
};

// GDX_TRACE=1: the timeline of search_host's chunks (start of the upload, kernels, end of the D2H) on stderr
struct Trace {
    struct Row {
        int k;
        uint64_t nq, bytes;
        EventPairs::Pair link, kernels;  // start of the upload .. end of the D2H; the kernels
        double host_stage_ms;
    };
    const bool on = [] {
        static const bool v = env_flag("GDX_TRACE", false);
        return v;
    }();
    const std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    EventPairs ev;
    EventPairs::Pair link = {};  // of the current chunk
    std::vector<Row> rows;
    void chunk_begins(cudaStream_t st) { if (on) cudaEventRecord((link = ev.next()).begin, st); }
    void kernels_recorded(int k, uint64_t nq, uint64_t bytes, const EventPairs::Pair &kernels, double stage_ms) {
        if (on) rows.push_back(Row{k, nq, bytes, link, kernels, stage_ms});
    }
    void d2h_recorded(cudaStream_t st) { if (on) cudaEventRecord(rows.back().link.end, st); }
    double ms() const {
        return on ? std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() : 0;
    }
    // once the streams have drained; t_issue: when the last chunk was issued
    void print(double t_issue) {
        if (rows.empty()) return;
        fprintf(stderr, "[gdx trace] host: all chunks issued at %.3f ms, streams drained at %.3f ms (%u pool threads)\n", t_issue,
                ms(), HostPool::get().threads());
        cudaEvent_t base = rows[0].link.begin;
        for (auto &r : rows) {
            float a = 0, b = 0, c = 0, d = 0;
            cudaError_t te = cudaEventElapsedTime(&a, base, r.link.begin);
            if (te != cudaSuccess) fprintf(stderr, "[gdx trace] elapsed: %s\n", cudaGetErrorString(te));
            cudaEventElapsedTime(&b, base, r.kernels.begin);
            cudaEventElapsedTime(&c, base, r.kernels.end);
            cudaEventElapsedTime(&d, base, r.link.end);
            fprintf(stderr, "[gdx trace] chunk %2d slot %d nq %8llu h2d bytes %10llu host stage %.3f ms | h2d %.3f..%.3f | kernels %.3f..%.3f | d2h ..%.3f\n",
                    r.k, r.k % kSlots, (unsigned long long)r.nq, (unsigned long long)r.bytes, r.host_stage_ms, a, b, b, c, d);
        }
    }
};

// uploads of a hybrid batch that may still be on the link, oldest first; each has left it once its slot's ev_link fired
struct LinkQueue {
    std::vector<std::pair<const Slot *, uint64_t>> q;  // (slot, bytes)
    cudaError_t push(Slot &sl, uint64_t bytes) {
        // this slot's event is about to be re-recorded: its older upload has long left the link
        q.erase(std::remove_if(q.begin(), q.end(), [&](const auto &u) { return u.first == &sl; }), q.end());
        q.emplace_back(&sl, bytes);
        return cudaEventRecord(sl.ev_link, sl.stream);
    }
    uint64_t backlog() {
        while (!q.empty() && cudaEventQuery(q.front().first->ev_link) == cudaSuccess) q.erase(q.begin());
        return std::accumulate(q.begin(), q.end(), 0ull, [](uint64_t b, const auto &u) { return b + u.second; });
    }
};

// The staging of search_host: per call, which caller buffers go through pinned staging and the packer's exception
// lists; per chunk, what stage_chunk made of it.
struct Staging {
    bool in, off;  // the symbols, the u64 offsets: pageable memory of a large batch
    bool off32;    // large variable-length batch: offsets cross chunk relative as u32 (chunks of < 2^32 symbols)
    std::vector<uint64_t> exc;    // symbol positions (chunk relative) the packer could not encode
    std::vector<uint32_t> exc_q;  // the queries (chunk relative) that hold them
    DevQueries dq, xq;  // the chunk; its queries with a byte without a 2-bit code (IO bytes, re-run into x_slots)
    const uint32_t *x_slots;
    bool packed;  // packed by the host
    double stage_ms;
    Uploads up;
};

// The uploads of one chunk on its slot's stream: its symbols (host-packed, pre-packed or IO bytes), its offsets (u32
// chunk relative or u64) and, for a host-packed chunk, the queries with a byte the packer has no code for.
gdx_status stage_chunk(const gdx_index *idx, const gdx_queries *qs, const gdx::Chunk &c, gdx::ChunkPlan &plan,
                       Slot &sl, Staging &u) {
    if (sl.h2d_pending) {  // the slot's staging buffers are free again once their last upload is done
        CUDA_TRY(cudaEventSynchronize(sl.ev_h2d));
        sl.h2d_pending = false;
    }
    const auto t0 = std::chrono::steady_clock::now();
    const uint64_t q0 = c.q0, cq = c.cq(), sym0 = c.sym0, nsym = c.nsym();
    u.xq = DevQueries{};
    u.packed = false;
    u.up = Uploads{sl.stream};
    if (nsym && c.pack) {
        CUDA_TRY(sl.h_in.reserve((nsym + 3) / 4 + 8));
        pack2_parallel(idx->pack, qs->bytes + sym0, nsym, (uint8_t *)sl.h_in.p, u.exc);
        gdx::exception_queries(qs->offsets, qs->fixed_len, q0, c.q1, sym0, u.exc, u.exc_q);
        u.packed = u.exc_q.size() * 16 <= cq;
        if (u.packed) CUDA_TRY(u.up.copy(sl.bytes.p, sl.h_in.p, (nsym + 3) / 4, &sl.h_in));
        else plan.packing_failed();
    }
    const bool words = u.packed || plan.prepacked;  // the kernel reads 2-bit words
    DevQueries &dq = u.dq = DevQueries{words ? nullptr : sl.bytes.as<uint8_t>(), nullptr, nullptr, qs->fixed_len, cq, 0, 0,
                                       words ? sl.bytes.as<uint32_t>() : nullptr, nsym};
    if (nsym && plan.prepacked) {  // the caller's stream, from the byte that holds the chunk's first symbol
        const uint64_t b0 = sym0 / 4, b1 = (c.sym1 + 3) / 4;
        CUDA_TRY(u.up.copy(sl.bytes.p, qs->bytes + b0, b1 - b0, u.in ? &sl.h_in : nullptr));
        dq.shift = sym0 & 3;
        dq.limit = nsym + dq.shift;
    } else if (nsym && !u.packed) {
        CUDA_TRY(u.up.copy(sl.bytes.p, qs->bytes + sym0, nsym, u.in ? &sl.h_in : nullptr));
    }
    if (qs->offsets && u.off32 && nsym + 4 < 0xffffffffull) {
        // chunk-relative 32-bit offsets, narrowed by the pool into pinned staging: half the PCIe bytes
        CUDA_TRY(sl.h_off.reserve((cq + 1) * 4));
        const uint64_t *osrc = qs->offsets + q0;
        uint32_t *o32 = (uint32_t *)sl.h_off.p;
        const uint64_t rel = sym0 - dq.shift, cnt = cq + 1;
        constexpr uint64_t kPiece = 1ull << 18;
        HostPool::get().parallel_for(div_up(cnt, kPiece), [&](uint64_t piece) {
            const uint64_t lo = piece * kPiece, hi = std::min(cnt, lo + kPiece);
            for (uint64_t i = lo; i < hi; ++i) o32[i] = (uint32_t)(osrc[i] - rel);
        });
        CUDA_TRY(u.up.copy(sl.offsets.p, o32, cnt * 4, &sl.h_off));
        dq.offsets32 = sl.offsets.as<uint32_t>();
        dq.shift = 0;
    } else if (qs->offsets) {
        CUDA_TRY(u.up.copy(sl.offsets.p, qs->offsets + q0, (cq + 1) * 8, u.off ? &sl.h_off : nullptr));
        dq.offsets = sl.offsets.as<uint64_t>();
        dq.base = sym0 - dq.shift;
        dq.shift = 0;
    }
    // queries with an exception byte: their offsets, result slots and IO bytes in one upload
    const uint64_t nx = u.packed ? u.exc_q.size() : 0;
    if (nx) {
        uint64_t xbytes = 0;
        for (uint32_t q : u.exc_q) xbytes += query_bytes_end(qs, q0 + q + 1) - query_bytes_end(qs, q0 + q);
        const uint64_t off_slots = (nx + 1) * 8, off_bytes = align_up(off_slots + nx * 4, 8), tot = off_bytes + xbytes + 8;
        GDX_TRY(reserve_drained(sl.stream, {{&sl.xbuf, tot}}));
        CUDA_TRY(sl.h_x.reserve(tot));
        uint64_t *xo = (uint64_t *)sl.h_x.p;
        uint32_t *xs = (uint32_t *)((uint8_t *)sl.h_x.p + off_slots);
        uint8_t *xb = (uint8_t *)sl.h_x.p + off_bytes;
        uint64_t acc = 0;
        for (uint64_t i = 0; i < nx; ++i) {
            xo[i] = acc;
            xs[i] = u.exc_q[i];
            acc += query_bytes_end(qs, q0 + xs[i] + 1) - query_bytes_end(qs, q0 + xs[i]);
        }
        xo[nx] = acc;
        constexpr uint64_t kPiece = 4096;  // queries per piece
        HostPool::get().parallel_for(div_up(nx, kPiece), [&](uint64_t piece) {
            const uint64_t lo = piece * kPiece, hi = std::min(nx, lo + kPiece);
            for (uint64_t i = lo; i < hi; ++i) {
                const uint64_t b0 = query_bytes_end(qs, q0 + xs[i]);
                memcpy(xb + xo[i], qs->bytes + b0, xo[i + 1] - xo[i]);
            }
        });
        CUDA_TRY(u.up.copy(sl.xbuf.p, sl.h_x.p, off_bytes + xbytes, &sl.h_x));
        u.xq = DevQueries{sl.xbuf.as<uint8_t>() + off_bytes, sl.xbuf.as<uint64_t>(), nullptr, 0, nx, 0, 0, nullptr, xbytes};
        u.x_slots = reinterpret_cast<const uint32_t *>(sl.xbuf.as<uint8_t>() + off_slots);
    }
    u.stage_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (u.up.staged) {
        CUDA_TRY(cudaEventRecord(sl.ev_h2d, sl.stream));
        sl.h2d_pending = true;
    }
    return GDX_OK;
}

// once search_host's streams have drained: its counters (device and host: io) into t_stats, error words into status
gdx_status search_result(Workspace *ws, const gdx_stats &io) {
    CUDA_TRY(ws->read_counters(ws->slot[0].stream));
    CUDA_TRY(cudaStreamSynchronize(ws->slot[0].stream));
    const Counters &cnt = *ws->cnt_h();
    t_stats.queries = io.queries;
    t_stats.packed_queries = io.packed_queries;
    t_stats.exception_queries = io.exception_queries;
    t_stats.h2d_bytes = io.h2d_bytes;
    t_stats.d2h_bytes += io.d2h_bytes;
    for (const Slot &s : ws->slot) {
        t_stats.kernel_ms_search += s.timing.elapsed_ms();
        t_stats.kernel_ms_locate += s.locate.timing.elapsed_ms();
    }
    t_stats.lf_steps = cnt.search.lf_steps;
    t_stats.walk_steps = cnt.search.verify_walk_steps + cnt.locate_walk_steps;
    t_stats.locate_walk_steps = cnt.locate_walk_steps;
    t_stats.verified_queries = cnt.search.verified_rows;
    return kernel_error(*std::min_element(cnt.err, cnt.err + kSlots),
                        "symbol in io representation should be valid (alphabet.rs:195-198)");
}

// Chunked pipeline over kSlots streams: stage / pack -> H2D(queries) -> k_search -> sink per chunk.  The sink (CountSink
// for counts and cursors, or LocatePipe) takes a chunk's results from the slot's out_a (out_b) in chunk() and completes
// the call in finish(); the slots' pinned h_out_a (h_out_b) are sized for sink.stage_elem bytes per result.
template <class Sink>
gdx_status search_host(const gdx_index *idx, Workspace *ws, const gdx_queries *qs, Sink &sink) {
    const uint64_t nq = qs->nq;
    // error words / counters are reset on slot 0's stream; the other slot streams (non-blocking: no implicit
    // ordering with anything) wait for that before their first kernel
    CUDA_TRY(ws->reset_counters(ws->slot[0].stream));
    CUDA_TRY(cudaEventRecord(ws->ev_a, ws->slot[0].stream));
    for (int s = 1; s < kSlots; ++s) CUDA_TRY(cudaStreamWaitEvent(ws->slot[s].stream, ws->ev_a, 0));
    Trace trace;
    const bool prepacked = qs->encoding == GDX_QUERIES_PACKED_2BIT;
    const uint64_t total_syms = query_bytes_end(qs, nq) - query_bytes_end(qs, 0);
    const uint64_t total_in = prepacked ? (total_syms + 3) / 4 : total_syms;
    // Ordinary (pageable) caller memory would make every cudaMemcpyAsync a blocking, driver-staged copy at
    // 8-14 GB/s.  Large batches are staged through the slots' own pinned buffers instead, filled by the host
    // thread pool; while they are staged, IO bytes of a <= 4-symbol alphabet are packed to 2 bits (a quarter
    // of the PCIe bytes) -- that pays for pinned caller buffers too.
    const bool pack = nq && !prepacked && idx->pack.usable && pack_enabled() && total_in >= kPackMinBytes;
    const bool src_pinned = nq && is_pinned(qs->bytes);
    Staging u{nq && total_in >= kStageMinBytes && !src_pinned,
              nq && qs->offsets && nq * 8 >= kStageMinBytes && !is_pinned(qs->offsets),
              qs->offsets && nq * 8 >= kStageMinBytes && narrow_enabled()};
    gdx::ChunkPlan plan{qs->offsets, qs->fixed_len, qs->first_symbol, nq, prepacked, pack, pack && src_pinned,
                        kChunkFirst, kChunkMax, kChunkTail, kChunkMaxQueries, 4.0e6 * HostPool::get().threads()};
    LinkQueue link;
    for (Slot &sl : ws->slot) sl.h2d_pending = false;
    // Large batches: size every slot once for the largest chunk this call can cut (the adaptive schedule cuts
    // different chunks in every call; growing a buffer in mid-flight means freeing it and a new
    // allocation, milliseconds each, with the streams drained).  The streams are idle here.
    if (nq && total_in >= kStageMinBytes) {
        const uint64_t max_sym = plan.max_chunk_symbols() + 64;
        const uint64_t max_q = qs->fixed_len ? std::min<uint64_t>(nq, max_sym / qs->fixed_len + 1) : 0;
        for (Slot &sl : ws->slot) {
            CUDA_TRY(sl.bytes.reserve(max_sym));
            if (pack) CUDA_TRY(sl.h_in.reserve(max_sym / 4 + 8));
            else if (u.in) CUDA_TRY(sl.h_in.reserve(std::min<uint64_t>(total_in, kChunkMax) + 64));
            CUDA_TRY(sl.out_a.reserve(max_q * 8));
            CUDA_TRY(sl.out_b.reserve(sink.writes_b ? max_q * 8 : 0));
            CUDA_TRY(sl.h_out_a.reserve(max_q * sink.stage_elem));
            CUDA_TRY(sl.h_out_b.reserve(sink.writes_b ? max_q * sink.stage_elem : 0));
        }
    }
    gdx_stats io = {nq};  // (queries)
    gdx::Chunk c;
    for (int k = 0; plan.next(c); ++k) {
        if (c.bad_offsets) return bad_offsets(c.q0);
        const uint64_t cq = c.cq();
        Slot &sl = ws->slot[k % kSlots];
        const SortPlan sp = plan_sort(idx, cq, qs->offsets ? 0 : qs->fixed_len);
        GDX_TRY(reserve_drained(sl.stream, {{&sl.bytes, c.nsym() + 64}, {&sl.offsets, qs->offsets ? (cq + 1) * 8 : 0},
                                            {&sl.out_a, cq * 8}, {&sl.out_b, sink.writes_b ? cq * 8 : 0},
                                            {&sl.sort, sp.use ? sp.total_bytes : 0}}));
        trace.chunk_begins(sl.stream);
        GDX_TRY(stage_chunk(idx, qs, c, plan, sl, u));
        const uint64_t sym_bytes = u.packed || prepacked ? (c.nsym() + 3) / 4 : c.nsym();
        if (plan.hybrid) {
            CUDA_TRY(link.push(sl, sym_bytes));
            plan.after_upload(u.packed, c.nsym(), u.stage_ms, u.packed ? link.backlog() : 0);
        }
        uint64_t *a = sl.out_a.as<uint64_t>(), *b = sink.writes_b ? sl.out_b.as<uint64_t>() : nullptr;
        const EventPairs::Pair ev = sl.timing.next();
        CUDA_TRY(cudaEventRecord(ev.begin, sl.stream));
        trace.kernels_recorded(k, cq, sym_bytes, ev, u.stage_ms);
        const uint32_t *perm = nullptr;
        if (sp.use) {
            GDX_TRY(sort_queries(idx, u.dq, sp, sl.sort.p, sl.stream, &perm));
            t_stats.kernel_launches += 2;
        }
        uint64_t *err = &ws->cnt_d()->err[k % kSlots];
        GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
            launch_search<decltype(L)>(idx, u.dq, a, b, sink.mode, sink.narrow, c.q0, err, &ws->cnt_d()->search, perm,
                                       nullptr, sl.stream);
            if (u.xq.nq)  // overwrites the slots of the queries the packed kernel could not see correctly
                launch_search<decltype(L)>(idx, u.xq, a, b, sink.mode, sink.narrow, c.q0, err, &ws->cnt_d()->search,
                                           nullptr, u.x_slots, sl.stream);
            return GDX_OK;
        }));
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(ev.end, sl.stream));
        if (u.packed || prepacked) io.packed_queries += cq;
        io.exception_queries += u.xq.nq;
        io.h2d_bytes += u.up.bytes;
        GDX_TRY(sink.chunk(sl, c.q0, cq));
        trace.d2h_recorded(sl.stream);
        t_stats.kernel_launches += 1 + (u.xq.nq ? 1 : 0);
    }
    GDX_TRY(sink.finish());
    const double t_issue = trace.ms();
    for (int s = 0; s < kSlots; ++s) CUDA_TRY(cudaStreamSynchronize(ws->slot[s].stream));
    trace.print(t_issue);
    io.d2h_bytes = sink.d2h;
    return search_result(ws, io);
}

gdx_status begin_call(const gdx_index *idx, const char *what) {
    if (!idx) return fail(GDX_ERR_BAD_ARG, "%s: idx is NULL", what);
    t_stats = gdx_stats{};
    return GDX_OK;
}

// CSR + expand + walk on device-resident intervals, on slot 0's stream; results in ws->locate (offsets: n + 1, hits)
gdx_status locate_device_intervals(const gdx_index *idx, Workspace *ws, const uint64_t *d_starts,
                                   const uint64_t *d_ends, uint64_t n, uint64_t *total_out) {
    cudaStream_t st = ws->slot[0].stream;
    IntervalHits &ih = ws->locate;
    const EventPairs::Pair ev = ih.timing.next();
    CUDA_TRY(cudaEventRecord(ev.begin, st));
    GDX_TRY(ih.count(st, d_starts, d_ends, n));
    CUDA_TRY(cudaEventSynchronize(ih.ev_total));
    const uint64_t total = ih.h()->hits;
    *total_out = total;
    if (total)
        GDX_TRY(ih.expand_walk(idx, st, d_starts, d_ends, n, total, ih.h()->wide, &ws->cnt_d()->locate_walk_steps, false));
    CUDA_TRY(cudaEventRecord(ev.end, st));
    return GDX_OK;
}

void release_pinned_hits(const gdx_index *idx, void *p) {
    std::lock_guard<std::mutex> lk(idx->mu);
    for (auto &b : idx->pinned)
        if (b.buf.p == p) b.in_use = false;
}

gdx_status acquire_pinned_hits(const gdx_index *idx, uint64_t bytes, void **out, uint64_t *cap_out = nullptr) {
    std::lock_guard<std::mutex> lk(idx->mu);
    PinnedHits *best = nullptr;
    for (auto &p : idx->pinned)
        if (!p.in_use && p.buf.bytes >= bytes && (!best || p.buf.bytes < best->buf.bytes)) best = &p;
    if (!best) {
        for (auto &p : idx->pinned)  // recycle the largest free but too small buffer
            if (!p.in_use && (!best || p.buf.bytes > best->buf.bytes)) best = &p;
        if (!best) {
            idx->pinned.emplace_back();
            best = &idx->pinned.back();
        }
        const uint64_t want = align_up(bytes + bytes / 4 + 4096, 4096);
        const cudaError_t e = best->buf.alloc(want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(GDX_ERR_OOM, "pinned host allocation of %llu bytes failed: %s", (unsigned long long)want,
                        cudaGetErrorString(e));
        }
    }
    best->in_use = true;
    *out = best->buf.p;
    if (cap_out) *cap_out = best->buf.bytes;
    return GDX_OK;
}

gdx_status finish_locate(const gdx_index *idx, Workspace *ws, uint64_t n, uint64_t total, uint64_t *hit_offsets,
                         gdx_hit **hits, uint64_t *num_hits) {
    cudaStream_t st = ws->slot[0].stream;
    void *h = nullptr;
    GDX_TRY(acquire_pinned_hits(idx, total * sizeof(gdx_hit), &h));
    const gdx_status copied = [&]() -> gdx_status {
        if (total) CUDA_TRY(cudaMemcpyAsync(h, ws->locate.hits.p, total * sizeof(gdx_hit), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(hit_offsets, ws->locate.offsets.p, (n + 1) * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ws->read_counters(st));
        CUDA_TRY(cudaStreamSynchronize(st));
        return GDX_OK;
    }();
    if (copied != GDX_OK) {
        cudaStreamSynchronize(st);
        release_pinned_hits(idx, h);
        return copied;
    }
    t_stats.kernel_ms_locate = ws->locate.timing.elapsed_ms();
    t_stats.hits = total;
    t_stats.walk_steps += ws->cnt_h()->locate_walk_steps;
    t_stats.locate_walk_steps = ws->cnt_h()->locate_walk_steps;
    *hits = (gdx_hit *)h;
    *num_hits = total;
    return GDX_OK;
}

}  // namespace

namespace {

// mode 0: cursors, 1: counts; elem: bytes per element of the caller's arrays
gdx_status search_many_impl(const gdx_index *idx, const gdx_queries *queries, void *a, void *b, uint32_t elem, int mode,
                            const char *what) {
    GDX_TRY(begin_call(idx, what));
    GDX_TRY(check_queries(idx, queries));
    if (queries->nq && (!a || (mode == 0 && !b))) return fail(GDX_ERR_BAD_ARG, "output is NULL");
    if (elem == 4 && idx->h.wide) return fail(GDX_ERR_UNSUPPORTED, "32-bit results need a text shorter than 2^32 symbols");
    return with_workspace(idx, [&](Workspace *ws) {
        CountSink sink(idx, queries->nq, a, b, elem, mode);
        return search_host(idx, ws, queries, sink);
    });
}

// write_last = false: hit_offsets[nq] is left alone (it is the first entry of the next shard's range)
// hit_counts != NULL: the compact form (gdx_hit32 hits, u32 hits per query, no offsets)
gdx_status locate_many_impl(const gdx_index *idx, const gdx_queries *queries, uint64_t *hit_offsets, gdx_hit **hits,
                            uint64_t *num_hits, bool write_last = true, uint32_t *hit_counts = nullptr) {
    GDX_TRY(begin_call(idx, "gdx_locate_many"));
    GDX_TRY(check_queries(idx, queries));
    if ((!hit_offsets && !hit_counts) || !hits || !num_hits) return fail(GDX_ERR_BAD_ARG, "output is NULL");
    *hits = nullptr;
    *num_hits = 0;
    if (hit_counts && (idx->h.wide || idx->h.ntexts > 0xffffffffull))
        return fail(GDX_ERR_UNSUPPORTED, "32-bit hits need a text shorter than 2^32 symbols");
    const uint64_t n = queries->nq;
    const uint64_t hit_bytes = hit_counts ? 8 : sizeof(gdx_hit);
    PinnedResult res{idx};
    const gdx_status st = with_workspace(idx, [&](Workspace *ws) -> gdx_status {
        // every chunk of the search pipeline carries on with counts -> scan -> expand -> walk -> D2H
        LocatePipe lp{idx, ws, res, hit_offsets};
        lp.hit_counts = hit_counts;
        lp.hit_bytes = hit_bytes;
        lp.stage_offsets =
            n * 8 >= kStageMinBytes && !is_pinned(hit_counts ? (const void *)hit_counts : (const void *)hit_offsets);
        GDX_TRY(acquire_pinned_hits(idx, std::max<uint64_t>(n, 4096) * hit_bytes, &res.p, &res.cap));
        return search_host(idx, ws, queries, lp);
    });
    if (st != GDX_OK) return st;
    const uint64_t total = res.used / hit_bytes;
    if (write_last && hit_offsets) hit_offsets[n] = total;
    t_stats.hits = total;
    *hits = (gdx_hit *)res.hand_over();
    *num_hits = total;
    return GDX_OK;
}

}  // namespace

extern "C" gdx_status gdx_cursors_many(const gdx_index *idx, const gdx_queries *queries, uint64_t *starts,
                                       uint64_t *ends) {
    return guarded([&] { return search_many_impl(idx, queries, starts, ends, 8, 0, "gdx_cursors_many"); });
}
extern "C" gdx_status gdx_cursors_many_u32(const gdx_index *idx, const gdx_queries *queries, uint32_t *starts,
                                           uint32_t *ends) {
    return guarded([&] { return search_many_impl(idx, queries, starts, ends, 4, 0, "gdx_cursors_many_u32"); });
}
extern "C" gdx_status gdx_count_many(const gdx_index *idx, const gdx_queries *queries, uint64_t *counts) {
    return guarded([&] { return search_many_impl(idx, queries, counts, nullptr, 8, 1, "gdx_count_many"); });
}
extern "C" gdx_status gdx_count_many_u32(const gdx_index *idx, const gdx_queries *queries, uint32_t *counts) {
    return guarded([&] { return search_many_impl(idx, queries, counts, nullptr, 4, 1, "gdx_count_many_u32"); });
}
extern "C" gdx_status gdx_locate_many(const gdx_index *idx, const gdx_queries *queries, uint64_t *hit_offsets,
                                      gdx_hit **hits, uint64_t *num_hits) {
    return guarded([&] { return locate_many_impl(idx, queries, hit_offsets, hits, num_hits); });
}

extern "C" gdx_status gdx_locate_many_compact(const gdx_index *idx, const gdx_queries *queries, uint32_t *hit_counts,
                                              gdx_hit32 **hits, uint64_t *num_hits) {
    return guarded([&]() -> gdx_status {
        if (!hit_counts) return fail(GDX_ERR_BAD_ARG, "output is NULL");
        return locate_many_impl(idx, queries, nullptr, reinterpret_cast<gdx_hit **>(hits), num_hits, true, hit_counts);
    });
}

extern "C" uint64_t gdx_packed_bytes(uint64_t total_symbols) { return align_up((total_symbols + 3) / 4, 4); }

extern "C" gdx_status gdx_pack_queries(const gdx_index *idx, const gdx_queries *q, uint8_t *packed_out,
                                       uint64_t *first_unencodable) {
    return guarded([&]() -> gdx_status {
        if (!idx || !packed_out) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        GDX_TRY(check_queries(idx, q));
        if (q->encoding != GDX_QUERIES_IO_BYTES) return fail(GDX_ERR_BAD_ARG, "the batch is already packed");
        if (!idx->pack.usable)
            return fail(GDX_ERR_UNSUPPORTED, "2-bit packing needs an alphabet with at most 4 searchable symbols (this one has %u)",
                        idx->h.ns);
        const uint64_t s0 = query_bytes_end(q, 0), s1 = query_bytes_end(q, q->nq);
        // symbols in front of the first query keep their place in the stream so that offsets stay valid
        const uint64_t nbytes = gdx_packed_bytes(s1);
        std::vector<uint64_t> exc;
        if (s0) memset(packed_out, 0, (s0 + 3) / 4);
        // the packer writes whole bytes: start on the byte that holds symbol s0 (codes before it belong to no query)
        const uint64_t a0 = s0 & ~3ull;
        pack2_parallel(idx->pack, q->bytes + a0, s1 - a0, packed_out + a0 / 4, exc);
        for (uint64_t i = (s1 + 3) / 4; i < nbytes; ++i) packed_out[i] = 0;
        uint64_t first = ~0ull;
        for (uint64_t pos : exc) {
            const uint64_t sym = a0 + pos;
            if (sym < s0) continue;
            first = q->offsets ? query_of_symbol(q->offsets, 0, q->nq + 1, sym) : (sym - q->first_symbol) / q->fixed_len;
            break;
        }
        if (first_unencodable) *first_unencodable = first;
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_pack_symbols(const gdx_alphabet *alphabet, const uint8_t *io_bytes, uint64_t n,
                                       uint8_t *packed_out, uint64_t *exception_positions, uint64_t capacity,
                                       uint64_t *num_exceptions) {
    return guarded([&]() -> gdx_status {
        if (!alphabet || (n && (!io_bytes || !packed_out))) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        GDX_TRY(validate_alphabet(*alphabet));
        PackTable t;
        build_pack_table(alphabet->io_to_dense, alphabet->num_searchable_dense_symbols, t);
        if (!t.usable) return fail(GDX_ERR_UNSUPPORTED, "2-bit packing needs an alphabet with at most 4 searchable symbols");
        std::vector<uint64_t> exc;
        pack2_parallel(t, io_bytes, n, packed_out, exc);
        if (num_exceptions) *num_exceptions = exc.size();
        for (uint64_t i = 0; i < exc.size() && i < capacity && exception_positions; ++i) exception_positions[i] = exc[i];
        return GDX_OK;
    });
}

// ================================================================================================
// one batch over several replicas
// ================================================================================================
extern "C" void gdx_shard_range(uint64_t n_items, uint32_t shard, uint32_t n_shards, uint64_t *begin, uint64_t *end) {
    // contiguous, balanced, order-preserving: the first n_items % n_shards shards get one item more
    if (n_shards == 0) n_shards = 1;
    if (shard > n_shards) shard = n_shards;
    const uint64_t base = n_items / n_shards, rem = n_items % n_shards;
    const uint64_t b = (uint64_t)shard * base + std::min<uint64_t>(shard, rem);
    if (begin) *begin = b;
    if (end) *end = shard >= n_shards ? b : b + base + (shard < rem ? 1 : 0);
}

namespace {

// the queries [b, e) of a batch as a batch of their own
gdx_queries sub_batch(const gdx_queries &q, uint64_t b, uint64_t e) {
    gdx_queries s = q;
    s.nq = e - b;
    if (q.offsets) {
        s.offsets = q.offsets + b;  // absolute stream positions: the symbol pointer stays
    } else {
        const uint64_t sym = (uint64_t)q.first_symbol + b * q.fixed_len;
        if (q.encoding == GDX_QUERIES_PACKED_2BIT) {
            s.bytes = q.bytes + sym / 4;
            s.first_symbol = (uint32_t)(sym & 3);
        } else {
            s.bytes = q.bytes + sym;
            s.first_symbol = 0;
        }
    }
    return s;
}

struct ShardResult {
    gdx_status st = GDX_OK;
    std::string error;
    uint64_t error_query = 0;
    gdx_stats stats = {};
};

// runs work(k, begin, end) for every local shard on its own host thread (shard 0 on the caller's) and merges
// status, error text and statistics into the caller's thread-local state
template <class F>
gdx_status run_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard, uint32_t n_shards,
                       const gdx_queries *queries, F &&work) {
    if (!replicas || n_local == 0 || n_shards == 0 || first_shard + n_local > n_shards)
        return fail(GDX_ERR_BAD_ARG, "bad shard arguments (n_local %u, first_shard %u, n_shards %u)", n_local, first_shard, n_shards);
    for (uint32_t k = 0; k < n_local; ++k) {
        if (!replicas[k]) return fail(GDX_ERR_BAD_ARG, "replica %u is NULL", k);
        const ImageHeader &h0 = replicas[0]->h, &hk = replicas[k]->h;
        if (hk.n != h0.n || hk.sigma != h0.sigma || hk.ns != h0.ns || hk.sampling_rate != h0.sampling_rate ||
            hk.lookup_depth != h0.lookup_depth || hk.ntexts != h0.ntexts)
            return fail(GDX_ERR_BAD_ARG, "replica %u is not a replica of replica 0", k);
    }
    GDX_TRY(check_queries(replicas[0], queries));
    std::vector<ShardResult> res(n_local);
    auto run = [&](uint32_t k) {
        const bool helps = HostPool::t_caller_helps;
        if (n_local > 1) HostPool::t_caller_helps = false;  // the pool alone does the staging work of all shards
        uint64_t b = 0, e = 0;
        gdx_shard_range(queries->nq, first_shard + k, n_shards, &b, &e);
        ShardResult &r = res[k];
        r.st = guarded([&] { return work(k, b, e); });
        if (r.st != GDX_OK) {
            r.error = t_error;
            r.error_query = b + t_error_query;
        }
        r.stats = t_stats;
        HostPool::t_caller_helps = helps;
    };
    std::vector<std::thread> threads;
    threads.reserve(n_local);
    uint32_t started = 1;
    try {
        for (; started < n_local; ++started) threads.emplace_back(run, started);
    } catch (const std::exception &) {  // could not start a thread: the shards without one run here, one after the other
    }
    run(0);
    for (uint32_t k = started; k < n_local; ++k) run(k);
    for (auto &t : threads) t.join();
    gdx_stats sum = {};
    gdx_status st = GDX_OK;
    for (uint32_t k = 0; k < n_local; ++k) {
        const gdx_stats &x = res[k].stats;
        sum.queries += x.queries;
        sum.lf_steps += x.lf_steps;
        sum.hits += x.hits;
        sum.walk_steps += x.walk_steps;
        sum.locate_walk_steps += x.locate_walk_steps;
        sum.kernel_launches += x.kernel_launches;
        sum.verified_queries += x.verified_queries;
        sum.packed_queries += x.packed_queries;
        sum.exception_queries += x.exception_queries;
        sum.h2d_bytes += x.h2d_bytes;
        sum.d2h_bytes += x.d2h_bytes;
        sum.kernel_ms_search = std::max(sum.kernel_ms_search, x.kernel_ms_search);  // the shards run side by side
        sum.kernel_ms_locate = std::max(sum.kernel_ms_locate, x.kernel_ms_locate);
        if (st == GDX_OK && res[k].st != GDX_OK) {  // the error of the lowest failing shard = the first offending query
            st = res[k].st;
            t_error = res[k].error;
            t_error_query = res[k].error_query;
        }
    }
    sum.shards = n_local;
    t_stats = sum;
    return st;
}

}  // namespace

extern "C" gdx_status gdx_count_many_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                             uint32_t n_shards, const gdx_queries *queries, uint64_t *counts) {
    return guarded([&] {
        return run_sharded(replicas, n_local, first_shard, n_shards, queries, [&](uint32_t k, uint64_t b, uint64_t e) {
            const gdx_queries sub = sub_batch(*queries, b, e);
            return search_many_impl(replicas[k], &sub, counts ? counts + b : nullptr, nullptr, 8, 1, "gdx_count_many_sharded");
        });
    });
}

extern "C" gdx_status gdx_cursors_many_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                               uint32_t n_shards, const gdx_queries *queries, uint64_t *starts,
                                               uint64_t *ends) {
    return guarded([&] {
        return run_sharded(replicas, n_local, first_shard, n_shards, queries, [&](uint32_t k, uint64_t b, uint64_t e) {
            const gdx_queries sub = sub_batch(*queries, b, e);
            return search_many_impl(replicas[k], &sub, starts ? starts + b : nullptr, ends ? ends + b : nullptr, 8, 0,
                                    "gdx_cursors_many_sharded");
        });
    });
}

extern "C" gdx_status gdx_locate_many_sharded_compact(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                                      uint32_t n_shards, const gdx_queries *queries, uint32_t *hit_counts,
                                                      gdx_hit32 **shard_hits, uint64_t *shard_num_hits) {
    return guarded([&]() -> gdx_status {
        if (!hit_counts || !shard_hits || !shard_num_hits) return fail(GDX_ERR_BAD_ARG, "output is NULL");
        for (uint32_t k = 0; k < n_local; ++k) {
            shard_hits[k] = nullptr;
            shard_num_hits[k] = 0;
        }
        gdx_status st = run_sharded(replicas, n_local, first_shard, n_shards, queries, [&](uint32_t k, uint64_t b, uint64_t e) {
            const gdx_queries sub = sub_batch(*queries, b, e);
            return locate_many_impl(replicas[k], &sub, nullptr, reinterpret_cast<gdx_hit **>(&shard_hits[k]), &shard_num_hits[k], true,
                                    hit_counts + b);
        });
        uint64_t total = 0;
        for (uint32_t k = 0; k < n_local; ++k) {
            if (st != GDX_OK && shard_hits[k]) {
                gdx_free_hits(replicas[k], reinterpret_cast<gdx_hit *>(shard_hits[k]));
                shard_hits[k] = nullptr;
                shard_num_hits[k] = 0;
            }
            total += shard_num_hits[k];
        }
        t_stats.hits = total;
        return st;
    });
}

extern "C" gdx_status gdx_locate_many_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                              uint32_t n_shards, const gdx_queries *queries, uint64_t *hit_offsets,
                                              gdx_hit **shard_hits, uint64_t *shard_first_hit) {
    return guarded([&]() -> gdx_status {
        if (!hit_offsets || !shard_hits || !shard_first_hit) return fail(GDX_ERR_BAD_ARG, "output is NULL");
        for (uint32_t k = 0; k < n_local; ++k) shard_hits[k] = nullptr;
        std::vector<uint64_t> n_hits(n_local, 0), begins(n_local, 0), ends(n_local, 0);
        // every shard writes its own CSR offsets (starting at 0) into its range of hit_offsets -- not the entry one
        // past the range, which is the next shard's first; the ranges are rebased below
        gdx_status st = run_sharded(replicas, n_local, first_shard, n_shards, queries, [&](uint32_t k, uint64_t b, uint64_t e) {
            const gdx_queries sub = sub_batch(*queries, b, e);
            begins[k] = b;
            ends[k] = e;
            return locate_many_impl(replicas[k], &sub, hit_offsets + b, &shard_hits[k], &n_hits[k], false);
        });
        if (st != GDX_OK) {
            for (uint32_t k = 0; k < n_local; ++k)
                if (shard_hits[k]) {
                    gdx_free_hits(replicas[k], shard_hits[k]);
                    shard_hits[k] = nullptr;
                }
            return st;
        }
        uint64_t acc = 0;
        for (uint32_t k = 0; k < n_local; ++k) {
            shard_first_hit[k] = acc;
            if (acc) {
                uint64_t *o = hit_offsets + begins[k];
                const uint64_t cnt = ends[k] - begins[k], base = acc;
                constexpr uint64_t kPiece = 1ull << 18;
                HostPool::get().parallel_for(div_up(cnt, kPiece), [&](uint64_t piece) {
                    const uint64_t lo = piece * kPiece, hi = std::min(cnt, lo + kPiece);
                    for (uint64_t i = lo; i < hi; ++i) o[i] += base;
                });
            }
            acc += n_hits[k];
        }
        shard_first_hit[n_local] = acc;
        hit_offsets[ends[n_local - 1]] = acc;
        t_stats.hits = acc;
        return GDX_OK;
    });
}

extern "C" gdx_status gdx_locate_intervals(const gdx_index *idx, const uint64_t *starts, const uint64_t *ends,
                                           uint64_t n, uint64_t *hit_offsets, gdx_hit **hits, uint64_t *num_hits) {
    return guarded([&]() -> gdx_status {
        GDX_TRY(begin_call(idx, "gdx_locate_intervals"));
        if (!hit_offsets || !hits || !num_hits || (n && (!starts || !ends))) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        *hits = nullptr;
        *num_hits = 0;
        for (uint64_t i = 0; i < n; ++i)
            if (starts[i] > ends[i] || ends[i] > idx->h.n)
                return fail(GDX_ERR_BAD_ARG, "interval %llu is not inside [0, text_len]", (unsigned long long)i);
        return with_workspace(idx, [&](Workspace *ws) -> gdx_status {
            cudaStream_t st = ws->slot[0].stream;
            CUDA_TRY(ws->starts.reserve((n + 1) * 8));
            CUDA_TRY(ws->ends.reserve((n + 1) * 8));
            CUDA_TRY(ws->reset_counters(st));
            if (n) {
                CUDA_TRY(cudaMemcpyAsync(ws->starts.p, starts, n * 8, cudaMemcpyHostToDevice, st));
                CUDA_TRY(cudaMemcpyAsync(ws->ends.p, ends, n * 8, cudaMemcpyHostToDevice, st));
            }
            uint64_t total = 0;
            GDX_TRY(locate_device_intervals(idx, ws, ws->starts.as<uint64_t>(), ws->ends.as<uint64_t>(), n, &total));
            return finish_locate(idx, ws, n, total, hit_offsets, hits, num_hits);
        });
    });
}

extern "C" void gdx_free_hits(const gdx_index *idx, gdx_hit *hits) {
    if (idx && hits) release_pinned_hits(idx, hits);
}

static gdx_status extend_many_on(const gdx_index *idx, Workspace *ws, uint64_t *starts, uint64_t *ends,
                                 const uint8_t *io_symbols, uint64_t n);

extern "C" gdx_status gdx_extend_many(const gdx_index *idx, uint64_t *starts, uint64_t *ends,
                                      const uint8_t *io_symbols, uint64_t n) {
    return guarded([&]() -> gdx_status {
        GDX_TRY(begin_call(idx, "gdx_extend_many"));
        if (n == 0) return GDX_OK;
        if (!starts || !ends || !io_symbols) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        return with_workspace(idx, [&](Workspace *ws) { return extend_many_on(idx, ws, starts, ends, io_symbols, n); });
    });
}

static gdx_status extend_many_on(const gdx_index *idx, Workspace *ws, uint64_t *starts, uint64_t *ends,
                                 const uint8_t *io_symbols, uint64_t n) {
    {
        cudaStream_t st = ws->slot[0].stream;
        CUDA_TRY(ws->starts.reserve(n * 8));
        CUDA_TRY(ws->ends.reserve(n * 8));
        CUDA_TRY(ws->symbols.reserve(n));
        CUDA_TRY(ws->reset_counters(st));
        CUDA_TRY(cudaStreamSynchronize(st));
        // large pageable cursor arrays go through pinned staging (see search_host)
        Slot &sl0 = ws->slot[0];
        const bool stage = n * 8 >= kStageMinBytes && !(is_pinned(starts) && is_pinned(ends));
        const uint64_t *src_s = starts, *src_e = ends;
        if (stage) {
            CUDA_TRY(sl0.h_out_a.reserve(n * 8));
            CUDA_TRY(sl0.h_out_b.reserve(n * 8));
            HostPool::get().copy(sl0.h_out_a.p, starts, n * 8);
            HostPool::get().copy(sl0.h_out_b.p, ends, n * 8);
            src_s = (const uint64_t *)sl0.h_out_a.p;
            src_e = (const uint64_t *)sl0.h_out_b.p;
        }
        uint64_t *d_s = ws->starts.as<uint64_t>(), *d_e = ws->ends.as<uint64_t>();
        uint8_t *d_c = ws->symbols.as<uint8_t>();
        // chunks of 1 M cursors round-robin over the workspace streams: upload, kernel and download of
        // neighbouring chunks overlap (PCIe is full duplex).  Results land in the staging buffers (pageable
        // caller arrays: handed over only on success) or directly in the caller's pinned arrays (on error their
        // contents are unspecified -- the reference panics in that case).
        const uint64_t kChunk = 1ull << 20;
        uint64_t launches = 0;
        for (uint64_t off = 0, k = 0; off < n; off += kChunk, ++k) {
            const uint64_t cn = std::min<uint64_t>(kChunk, n - off);
            cudaStream_t cs = ws->slot[k % kSlots].stream;
            CUDA_TRY(cudaMemcpyAsync(d_s + off, src_s + off, cn * 8, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_e + off, src_e + off, cn * 8, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_c + off, io_symbols + off, cn, cudaMemcpyHostToDevice, cs));
            GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
                k_extend<decltype(L)><<<(unsigned)div_up(cn, 256), 256, 0, cs>>>(idx->dev, d_s + off, d_e + off, d_c + off, cn,
                                                                               &ws->cnt_d()->extend_bad_symbol, off);
                return GDX_OK;
            }));
            CUDA_TRY(cudaGetLastError());
            ++launches;
            uint64_t *dst_s = stage ? (uint64_t *)sl0.h_out_a.p : starts, *dst_e = stage ? (uint64_t *)sl0.h_out_b.p : ends;
            CUDA_TRY(cudaMemcpyAsync(dst_s + off, d_s + off, cn * 8, cudaMemcpyDeviceToHost, cs));
            CUDA_TRY(cudaMemcpyAsync(dst_e + off, d_e + off, cn * 8, cudaMemcpyDeviceToHost, cs));
        }
        for (int s2 = 0; s2 < kSlots; ++s2) CUDA_TRY(cudaStreamSynchronize(ws->slot[s2].stream));
        CUDA_TRY(ws->read_counters(st));
        CUDA_TRY(cudaStreamSynchronize(st));
        t_stats.kernel_launches = launches;
        const Counters &c = *ws->cnt_h();
        if (c.extend_bad_cursor != kNoError)  // checked on the device: text_with_rank_support/mod.rs:106-110
            return fail(GDX_ERR_BAD_ARG, "cursor %llu is outside [0, text_len]", (unsigned long long)c.extend_bad_cursor);
        if (c.extend_bad_symbol != kNoError) {
            t_error_query = c.extend_bad_symbol;
            return fail(GDX_ERR_INVALID_SYMBOL, "cursor %llu: symbol in io representation should be valid (alphabet.rs:195-198)",
                        (unsigned long long)c.extend_bad_symbol);
        }
        if (stage) {
            HostPool::get().copy(starts, sl0.h_out_a.p, n * 8);
            HostPool::get().copy(ends, sl0.h_out_b.p, n * 8);
        }
        return GDX_OK;
    }
}

extern "C" gdx_status gdx_cursor_for_query(const gdx_index *idx, const uint8_t *query, uint64_t len, uint64_t *start,
                                           uint64_t *end) {
    return guarded([&]() -> gdx_status {
        if (!idx || !start || !end || (len && !query)) return fail(GDX_ERR_BAD_ARG, "NULL argument");
        // single-query path of the reference (lib.rs:217-235): when the lookup-table interval is already
        // empty, the next symbol to the left is still translated (and may panic) before the loop breaks.
        const uint32_t D = idx->h.lookup_depth;
        gdx_queries q = {query, nullptr, len, 1};
        uint8_t dummy = 0;
        if (len == 0) q.bytes = &dummy;
        gdx_status st = gdx_cursors_many(idx, &q, start, end);
        if (st != GDX_OK) return st;
        if (D > 0 && len > D && *start == *end) {
            gdx_queries suffix = {query + (len - D), nullptr, D, 1};
            uint64_t s2 = 0, e2 = 0;
            GDX_TRY(gdx_cursors_many(idx, &suffix, &s2, &e2));
            if (s2 == e2 && idx->h.io_to_dense[query[len - D - 1]] == 0) {
                t_error_query = 0;
                return fail(GDX_ERR_INVALID_SYMBOL, "symbol in io representation should be valid (alphabet.rs:195-198)");
            }
        }
        return GDX_OK;
    });
}

// ================================================================================================
// Hamming search (no counterpart in the reference; semantics in include/genedex_b200.h, search in hamming.h)
// ================================================================================================
namespace {

static_assert(sizeof(HammingInterval) == sizeof(gdx_hamming_interval), "HammingInterval mirrors gdx_hamming_interval");
static_assert(GDX_HAMMING_MAX_MISMATCHES == kHammingMaxMismatches && GDX_HAMMING_MAX_QUERY_LEN == kHammingMaxQueryLen,
              "hamming.h and the header agree on the limits");

// queries per chunk: bounds the workspace (query bytes, per-query counts and offsets) whatever the batch size,
// while one chunk still puts a thread on every slot of the device
constexpr uint64_t kHammingChunkQueries = 1ull << 20;

enum HammingMode { kHammingCount = 0, kHammingCursors = 1, kHammingLocate = 2 };

// The first query the host refuses, nq if none: offsets that decrease or leave [offsets[0], offsets[nq]]
// (GDX_ERR_BAD_ARG) or a query longer than GDX_HAMMING_MAX_QUERY_LEN (GDX_ERR_UNSUPPORTED).  One pass over the
// offsets, which is cheap next to a search that may branch at every symbol.
uint64_t hamming_host_check(const gdx_queries *q, gdx_status *st) {
    *st = GDX_OK;
    if (q->nq == 0) return 0;
    if (!q->offsets) {
        if (q->fixed_len <= kHammingMaxQueryLen) return q->nq;
        *st = GDX_ERR_UNSUPPORTED;
        return 0;
    }
    const uint64_t lo = q->offsets[0], hi = q->offsets[q->nq];
    for (uint64_t i = 0; i < q->nq; ++i) {
        const uint64_t b = q->offsets[i], e = q->offsets[i + 1];
        if (e < b || b < lo || e > hi) {
            *st = GDX_ERR_BAD_ARG;
            return i;
        }
        if (e - b > kHammingMaxQueryLen) {
            *st = GDX_ERR_UNSUPPORTED;
            return i;
        }
    }
    return q->nq;
}

constexpr const char *kHammingBadSymbol = "every byte of a Hamming query must be a searchable symbol";

// Chunks of kHammingChunkQueries over the queries [0, n_ok) on slot 0's stream: upload -> pass 1 (checks + counts)
// -> [scan -> pass 2 (intervals) -> locate] -> results to the caller.  counts == NULL in kHammingCount mode: only
// check the queries (an error is then looked for in front of a query the host refused).  The per-query CSR lives in
// slot 0's IntervalHits (used as scratch only), the locate of the intervals in the workspace's.
gdx_status hamming_run(const gdx_index *idx, Workspace *ws, const gdx_queries *qs, uint32_t k, int mode, uint64_t n_ok,
                       uint64_t *counts, uint64_t *offsets_out, PinnedResult &res) {
    Slot &sl = ws->slot[0];
    IntervalHits &csr = sl.locate;
    cudaStream_t st = sl.stream;
    const uint64_t strata = k + 1;
    const uint64_t elem = mode == kHammingCursors ? sizeof(gdx_hamming_interval) : sizeof(gdx_hit);
    uint64_t *d_err = &ws->cnt_d()->err[0];
    CUDA_TRY(ws->reset_counters(st));
    const bool src_pinned = n_ok && is_pinned(qs->bytes);
    Uploads up{st};
    uint64_t d2h = 0, launches = 0;
    for (uint64_t q0 = 0; q0 < n_ok; q0 += kHammingChunkQueries) {
        const uint64_t cq = std::min<uint64_t>(kHammingChunkQueries, n_ok - q0);
        const uint64_t sym0 = query_bytes_end(qs, q0), nsym = query_bytes_end(qs, q0 + cq) - sym0;
        // the chunk's IO bytes (pageable: through pinned staging) + offsets (staged); the previous chunk's copies are done
        CUDA_TRY(sl.bytes.reserve(nsym + 8));
        if (nsym) CUDA_TRY(up.copy(sl.bytes.p, qs->bytes + sym0, nsym, src_pinned ? nullptr : &sl.h_in));
        DevQueries dq = {};
        dq.bytes = sl.bytes.as<uint8_t>();
        dq.fixed_len = qs->fixed_len;
        dq.nq = cq;
        dq.limit = nsym;
        if (qs->offsets) {
            CUDA_TRY(sl.offsets.reserve((cq + 1) * 8));
            CUDA_TRY(up.copy(sl.offsets.p, qs->offsets + q0, (cq + 1) * 8, &sl.h_off));
            dq.offsets = sl.offsets.as<uint64_t>();
            dq.base = sym0;
        }
        // pass 1: checks, per-stratum counts, intervals per query
        const bool intervals = mode != kHammingCount;
        CUDA_TRY(sl.out_a.reserve(cq * strata * 8));
        if (intervals) {
            CUDA_TRY(csr.counts.reserve((cq + 1) * 8));
            CUDA_TRY(csr.offsets.reserve((cq + 1) * 8));
            CUDA_TRY(cudaMemsetAsync(csr.counts.as<uint64_t>() + cq, 0, 8, st));
        }
        const unsigned grid = (unsigned)div_up(cq, 256);
        const EventPairs::Pair ev = sl.timing.next();
        CUDA_TRY(cudaEventRecord(ev.begin, st));
        GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
            k_hamming<decltype(L), 1><<<grid, 256, 0, st>>>(idx->dev, dq, k, q0, d_err, sl.out_a.as<uint64_t>(),
                                                             intervals ? csr.counts.as<uint64_t>() : nullptr, nullptr,
                                                             nullptr, nullptr, &ws->cnt_d()->hamming_expansions);
            return GDX_OK;
        }));
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(ev.end, st));
        ++launches;
        if (!intervals) {
            if (counts) {
                CUDA_TRY(sl.h_out_a.reserve(cq * strata * 8));
                CUDA_TRY(cudaMemcpyAsync(sl.h_out_a.p, sl.out_a.p, cq * strata * 8, cudaMemcpyDeviceToHost, st));
                d2h += cq * strata * 8;
            }
            CUDA_TRY(ws->read_counters(st));
            CUDA_TRY(cudaStreamSynchronize(st));
            GDX_TRY(kernel_error(ws->cnt_h()->err[0], kHammingBadSymbol));
            if (counts) HostPool::get().copy(counts + q0 * strata, sl.h_out_a.p, cq * strata * 8);
            continue;
        }
        // CSR of the chunk's intervals
        GDX_TRY(exclusive_sum(csr.scan_tmp, csr.counts.as<uint64_t>(), csr.offsets.as<uint64_t>(), cq + 1, st));
        CUDA_TRY(ws->read_counters(st));
        CUDA_TRY(cudaMemcpyAsync(&csr.h()->hits, csr.offsets.as<uint64_t>() + cq, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        ++launches;
        GDX_TRY(kernel_error(ws->cnt_h()->err[0], kHammingBadSymbol));
        const uint64_t niv = csr.h()->hits;
        // pass 2: the intervals at their CSR offsets in search order, a sort by start within every query, then records
        // (cursors) or starts / ends (the locate path)
        const uint64_t rec_bytes = mode == kHammingCursors ? sizeof(HammingInterval) : 8;
        const uint64_t held = csr.rows.bytes + csr.wide.bytes + ws->starts.bytes + sl.xbuf.bytes +
                              (mode == kHammingCursors ? csr.hits.bytes : ws->ends.bytes);
        const uint64_t need = niv * (32 + rec_bytes);
        bool fits = niv <= 0x7fffffffull;  // (the segmented sort counts items in an int)
        if (fits && need > held) {
            size_t free_b = 0, total_b = 0;
            CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
            fits = need <= free_b + held;
        }
        if (!fits)
            return fail(GDX_ERR_OOM, "%llu intervals of one chunk do not fit into device memory; split the batch",
                        (unsigned long long)niv);
        const uint64_t nr = std::max<uint64_t>(niv, 1);
        CUDA_TRY(csr.rows.reserve(nr * 8));
        CUDA_TRY(csr.wide.reserve(nr * 8));
        CUDA_TRY(ws->starts.reserve(nr * 8));
        CUDA_TRY(sl.xbuf.reserve(nr * 8));
        CUDA_TRY(mode == kHammingCursors ? csr.hits.reserve(nr * rec_bytes) : ws->ends.reserve(nr * 8));
        if (niv) {
            const EventPairs::Pair ev2 = sl.timing.next();
            CUDA_TRY(cudaEventRecord(ev2.begin, st));
            GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
                k_hamming<decltype(L), 2><<<grid, 256, 0, st>>>(idx->dev, dq, k, q0, nullptr, nullptr, nullptr,
                                                                 csr.offsets.as<uint64_t>(), csr.rows.as<uint64_t>(),
                                                                 csr.wide.as<uint64_t>(), nullptr);
                return GDX_OK;
            }));
            CUDA_TRY(cudaGetLastError());
            size_t sort_tmp = 0;
            const uint64_t *seg = csr.offsets.as<uint64_t>();
            CUDA_TRY(cub::DeviceSegmentedSort::SortPairs(nullptr, sort_tmp, csr.rows.as<uint64_t>(), ws->starts.as<uint64_t>(),
                                                         csr.wide.as<uint64_t>(), sl.xbuf.as<uint64_t>(), (int)niv, (int)cq,
                                                         seg, seg + 1, st));
            CUDA_TRY(sl.sort.reserve(sort_tmp));
            CUDA_TRY(cub::DeviceSegmentedSort::SortPairs(sl.sort.p, sort_tmp, csr.rows.as<uint64_t>(), ws->starts.as<uint64_t>(),
                                                         csr.wide.as<uint64_t>(), sl.xbuf.as<uint64_t>(), (int)niv, (int)cq,
                                                         seg, seg + 1, st));
            k_hamming_decode<<<(unsigned)div_up(niv, 256), 256, 0, st>>>(
                ws->starts.as<uint64_t>(), sl.xbuf.as<uint64_t>(), niv,
                mode == kHammingCursors ? csr.hits.as<HammingInterval>() : nullptr,
                mode == kHammingCursors ? nullptr : ws->ends.as<uint64_t>());
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaEventRecord(ev2.end, st));
            launches += 3;
        }
        // results of the chunk: records (cursors) or hits (locate, the walk of gdx_locate_intervals) + per-query offsets
        uint64_t n_out = niv;
        const uint64_t *d_query_off = csr.offsets.as<uint64_t>();
        if (mode == kHammingLocate) {
            GDX_TRY(locate_device_intervals(idx, ws, ws->starts.as<uint64_t>(), ws->ends.as<uint64_t>(), niv, &n_out));
            CUDA_TRY(sl.out_b.reserve(cq * 8));
            k_gather_u64<<<grid, 256, 0, st>>>(csr.offsets.as<uint64_t>(), ws->locate.offsets.as<uint64_t>(), cq,
                                               sl.out_b.as<uint64_t>());
            CUDA_TRY(cudaGetLastError());
            ++launches;
            d_query_off = sl.out_b.as<uint64_t>();
        }
        const uint64_t base = res.used / elem;
        GDX_TRY(res.reserve(res.used + n_out * elem));
        if (n_out) {
            const void *d_src = mode == kHammingCursors ? csr.hits.p : ws->locate.hits.p;
            CUDA_TRY(cudaMemcpyAsync((uint8_t *)res.p + res.used, d_src, n_out * elem, cudaMemcpyDeviceToHost, st));
            d2h += n_out * elem;
        }
        CUDA_TRY(sl.h_out_a.reserve(cq * 8));
        CUDA_TRY(cudaMemcpyAsync(sl.h_out_a.p, d_query_off, cq * 8, cudaMemcpyDeviceToHost, st));
        d2h += cq * 8;
        CUDA_TRY(cudaStreamSynchronize(st));
        const uint64_t *h_off = (const uint64_t *)sl.h_out_a.p;
        for (uint64_t i = 0; i < cq; ++i) offsets_out[q0 + i] = base + h_off[i];
        res.used += n_out * elem;
    }
    CUDA_TRY(ws->read_counters(st));
    CUDA_TRY(cudaStreamSynchronize(st));
    t_stats.queries = qs->nq;
    t_stats.lf_steps = ws->cnt_h()->hamming_expansions;
    t_stats.kernel_ms_search = sl.timing.elapsed_ms();
    t_stats.kernel_ms_locate = ws->locate.timing.elapsed_ms();
    t_stats.kernel_launches += launches;
    t_stats.h2d_bytes = up.bytes;
    t_stats.d2h_bytes = d2h;
    if (mode == kHammingLocate) t_stats.hits = res.used / elem;
    return GDX_OK;
}

gdx_status hamming_many_impl(const gdx_index *idx, const gdx_queries *queries, uint32_t k, int mode, uint64_t *counts,
                             uint64_t *offsets_out, void **result, uint64_t *num_out, const char *what) {
    GDX_TRY(begin_call(idx, what));
    GDX_TRY(check_queries(idx, queries));
    if (k > GDX_HAMMING_MAX_MISMATCHES)
        return fail(GDX_ERR_BAD_ARG, "%s: max_mismatches %u is larger than GDX_HAMMING_MAX_MISMATCHES (%d)", what, k,
                    GDX_HAMMING_MAX_MISMATCHES);
    if (queries->encoding != GDX_QUERIES_IO_BYTES)
        return fail(GDX_ERR_UNSUPPORTED, "%s takes IO-byte queries (GDX_QUERIES_IO_BYTES) only", what);
    if (mode == kHammingCount ? (queries->nq && !counts) : (!offsets_out || !result || !num_out))
        return fail(GDX_ERR_BAD_ARG, "output is NULL");
    if (result) {
        *result = nullptr;
        *num_out = 0;
    }
    gdx_status host_st = GDX_OK;
    const uint64_t n_ok = hamming_host_check(queries, &host_st);
    PinnedResult res{idx};
    const gdx_status st = with_workspace(idx, [&](Workspace *ws) -> gdx_status {
        if (mode != kHammingCount) GDX_TRY(res.reserve(4096));
        // with a query the host refuses, the queries in front of it are only checked: a smaller offender wins
        if (host_st == GDX_OK) return hamming_run(idx, ws, queries, k, mode, n_ok, counts, offsets_out, res);
        GDX_TRY(hamming_run(idx, ws, queries, k, kHammingCount, n_ok, nullptr, nullptr, res));
        if (host_st == GDX_ERR_BAD_ARG) return bad_offsets(n_ok);
        t_error_query = n_ok;
        return fail(GDX_ERR_UNSUPPORTED, "query %llu is longer than GDX_HAMMING_MAX_QUERY_LEN (%d symbols)",
                    (unsigned long long)n_ok, GDX_HAMMING_MAX_QUERY_LEN);
    });
    if (st != GDX_OK) return st;
    if (mode != kHammingCount) {
        const uint64_t elem = mode == kHammingCursors ? sizeof(gdx_hamming_interval) : sizeof(gdx_hit);
        offsets_out[queries->nq] = res.used / elem;
        *result = res.hand_over();
        *num_out = res.used / elem;
    }
    return GDX_OK;
}

}  // namespace

extern "C" gdx_status gdx_count_many_hamming(const gdx_index *idx, const gdx_queries *queries, uint32_t max_mismatches,
                                             uint64_t *counts) {
    return guarded([&] {
        return hamming_many_impl(idx, queries, max_mismatches, kHammingCount, counts, nullptr, nullptr, nullptr,
                                 "gdx_count_many_hamming");
    });
}
extern "C" gdx_status gdx_cursors_many_hamming(const gdx_index *idx, const gdx_queries *queries, uint32_t max_mismatches,
                                               uint64_t *interval_offsets, gdx_hamming_interval **intervals,
                                               uint64_t *num_intervals) {
    return guarded([&] {
        return hamming_many_impl(idx, queries, max_mismatches, kHammingCursors, nullptr, interval_offsets,
                                 reinterpret_cast<void **>(intervals), num_intervals, "gdx_cursors_many_hamming");
    });
}
extern "C" gdx_status gdx_locate_many_hamming(const gdx_index *idx, const gdx_queries *queries, uint32_t max_mismatches,
                                              uint64_t *hit_offsets, gdx_hit **hits, uint64_t *num_hits) {
    return guarded([&] {
        return hamming_many_impl(idx, queries, max_mismatches, kHammingLocate, nullptr, hit_offsets,
                                 reinterpret_cast<void **>(hits), num_hits, "gdx_locate_many_hamming");
    });
}

// ================================================================================================
// device-resident entry points
// ================================================================================================
static gdx_status search_device(const gdx_index *idx, const gdx_queries *dq_in, uint64_t *a, uint64_t *b, int mode,
                                uint64_t *d_error, void *stream) {
    if (!idx || !dq_in) return fail(GDX_ERR_BAD_ARG, "NULL argument");
    DeviceGuard guard(idx->device);
    // (offsets is a device pointer here: nothing of the batch may be dereferenced on the host)
    if (dq_in->encoding > GDX_QUERIES_PACKED_2BIT) return fail(GDX_ERR_BAD_ARG, "unknown queries->encoding %u", dq_in->encoding);
    if (dq_in->encoding == GDX_QUERIES_PACKED_2BIT && idx->h.ns > 4)
        return fail(GDX_ERR_UNSUPPORTED, "2-bit packed queries need an alphabet with at most 4 searchable symbols");
    DevQueries dq;
    const bool packed = dq_in->encoding == GDX_QUERIES_PACKED_2BIT;
    if (packed && (reinterpret_cast<uintptr_t>(dq_in->bytes) & 3u))
        return fail(GDX_ERR_BAD_ARG, "a packed device batch must be 4-byte aligned (and a multiple of 4 bytes long)");
    dq.bytes = packed ? nullptr : dq_in->bytes;
    dq.packed = packed ? reinterpret_cast<const uint32_t *>(dq_in->bytes) : nullptr;
    dq.offsets = dq_in->offsets;
    dq.offsets32 = nullptr;
    dq.fixed_len = dq_in->fixed_len;
    dq.nq = dq_in->nq;
    dq.base = 0;
    dq.shift = dq_in->first_symbol;
    dq.limit = ~0ull;  // device-resident batch: its extent is the caller's contract (header)
    cudaStream_t st = (cudaStream_t)stream;
    const SortPlan sp = plan_sort(idx, dq.nq, dq.offsets ? 0 : dq.fixed_len);
    const uint32_t *perm = nullptr;
    AsyncMem scratch;
    if (sp.use) {  // stream-ordered scratch from the device's memory pool
        CUDA_TRY(scratch.alloc(sp.total_bytes, st));
        GDX_TRY(sort_queries(idx, dq, sp, scratch.p, st, &perm));
    }
    GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
        launch_search<decltype(L)>(idx, dq, a, b, mode, false, 0, d_error, nullptr, perm, nullptr, st);
        return GDX_OK;
    }));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(scratch.free());
    return GDX_OK;
}

extern "C" gdx_status gdx_cursors_many_device(const gdx_index *idx, const gdx_queries *d_queries, uint64_t *d_starts,
                                              uint64_t *d_ends, uint64_t *d_error, void *stream) {
    return guarded([&] { return search_device(idx, d_queries, d_starts, d_ends, 0, d_error, stream); });
}
extern "C" gdx_status gdx_count_many_device(const gdx_index *idx, const gdx_queries *d_queries, uint64_t *d_counts,
                                            uint64_t *d_error, void *stream) {
    return guarded([&] { return search_device(idx, d_queries, d_counts, nullptr, 1, d_error, stream); });
}

extern "C" gdx_status gdx_locate_intervals_device(const gdx_index *idx, const uint64_t *d_starts,
                                                  const uint64_t *d_ends, uint64_t n, const uint64_t *d_hit_offsets,
                                                  uint64_t num_hits, gdx_hit *d_hits, void *stream) {
    if (!idx) return fail(GDX_ERR_BAD_ARG, "idx is NULL");
    if (n == 0 || num_hits == 0) return GDX_OK;
    if (!d_starts || !d_ends || !d_hit_offsets || !d_hits) return fail(GDX_ERR_BAD_ARG, "NULL argument");
    DeviceGuard guard(idx->device);
    cudaStream_t st = (cudaStream_t)stream;
    // stream-ordered scratch: rows (8 B per hit), worklist of wide intervals, two counters
    AsyncMem rows_mem, big_mem;
    CUDA_TRY(rows_mem.alloc(num_hits * 8, st));
    CUDA_TRY(big_mem.alloc((n + 2) * 8, st));
    uint64_t *rows = rows_mem.as<uint64_t>(), *big = big_mem.as<uint64_t>();
    CUDA_TRY(cudaMemsetAsync(big, 0, 16, st));
    k_expand_rows<<<(unsigned)div_up(n, 256), 256, 0, st>>>(d_starts, d_ends, d_hit_offsets, n, rows, big + 2,
                                                           reinterpret_cast<unsigned long long *>(big));
    CUDA_TRY(cudaGetLastError());
    uint64_t nbig = 0;  // the number of wide intervals decides the next grid: one small D2H + sync
    CUDA_TRY(cudaMemcpyAsync(&nbig, big, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (nbig) {
        dim3 grid((unsigned)nbig, 32);
        k_expand_big_rows<<<grid, 256, 0, st>>>(d_starts, d_ends, d_hit_offsets, big + 2, rows);
    }
    GDX_TRY(dispatch_layout(idx->h.layout, [&](auto L) -> gdx_status {
        launch_locate_walk<decltype(L)>(idx, rows, num_hits, reinterpret_cast<ulonglong2 *>(d_hits), nullptr, st);
        return GDX_OK;
    }));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(rows_mem.free());
    CUDA_TRY(big_mem.free());
    return GDX_OK;
}

// ================================================================================================
// random-gather ceiling
// ================================================================================================
__global__ void k_fill_random(uint64_t *p, uint64_t nwords) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords;
         i += (uint64_t)gridDim.x * blockDim.x)
        p[i] = mix64(i);
}

extern "C" gdx_status gdx_measure_random_gather(int32_t device_req, uint64_t table_bytes, uint32_t record_bytes,
                                                uint64_t loads, int32_t chained, double *gbps_out,
                                                double *gloads_out) {
    if (record_bytes != 32 && record_bytes != 64 && record_bytes != 128)
        return fail(GDX_ERR_BAD_ARG, "record_bytes must be 32, 64 or 128");
    int device;
    GDX_TRY(resolve_device(device_req, &device));
    DeviceGuard guard(device);
    uint64_t nrec = 1;
    while (nrec * 2 * record_bytes <= table_bytes) nrec *= 2;
    DevMem table_mem, sink_mem;
    CUDA_TRY(table_mem.alloc(nrec * record_bytes));
    auto check = [](cudaError_t e) {
        return e == cudaSuccess ? GDX_OK : fail(GDX_ERR_CUDA, "gather microbenchmark failed: %s", cudaGetErrorString(e));
    };
    GDX_TRY(check(sink_mem.alloc(8)));
    const uint8_t *table = table_mem.as<uint8_t>();
    uint64_t *sink = sink_mem.as<uint64_t>();
    Event e0, e1;
    float ms = 0;
    const unsigned blocks = 148 * 8, threads = 256;
    uint32_t rounds = (uint32_t)std::max<uint64_t>(1, loads / (2ull * blocks * threads));
    auto launch = [&](uint32_t r) {
        if (record_bytes == 32) k_gather<32><<<blocks, threads>>>(table, nrec - 1, r, chained, sink);
        else if (record_bytes == 64) k_gather<64><<<blocks, threads>>>(table, nrec - 1, r, chained, sink);
        else k_gather<128><<<blocks, threads>>>(table, nrec - 1, r, chained, sink);
    };
    k_fill_random<<<blocks, threads>>>(table_mem.as<uint64_t>(), nrec * record_bytes / 8);
    launch(rounds / 8 + 1);  // warm-up
    GDX_TRY(check(e0.create(cudaEventDefault)));
    GDX_TRY(check(e1.create(cudaEventDefault)));
    GDX_TRY(check(cudaEventRecord(e0)));
    launch(rounds);
    GDX_TRY(check(cudaEventRecord(e1)));
    GDX_TRY(check(cudaEventSynchronize(e1)));
    GDX_TRY(check(cudaEventElapsedTime(&ms, e0, e1)));
    const double nloads = 2.0 * blocks * threads * (double)rounds;
    if (gloads_out) *gloads_out = nloads / (ms * 1e-3) / 1e9;
    if (gbps_out) *gbps_out = nloads * record_bytes / (ms * 1e-3) / 1e9;
    return GDX_OK;
}
