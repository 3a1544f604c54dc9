// How the host pipeline of api.cu (search_host) cuts a batch into chunks.  Host only and free of CUDA, so that the
// schedule runs on the CPU against a plain model (tests/test_chunk_plan_host.py).
#pragma once
#include <algorithm>
#include <cstdint>
#include <vector>

namespace gdx {

// the last index i in [lo, hi) with offsets[i] <= sym, lo - 1 if there is none: for sorted offsets the query that holds
// symbol sym
inline uint64_t query_of_symbol(const uint64_t *offsets, uint64_t lo, uint64_t hi, uint64_t sym) {
    return (uint64_t)(std::upper_bound(offsets + lo, offsets + hi, sym) - offsets) - 1;
}

// The queries of chunk [q0, q1) (chunk relative, a run of one query once) that hold the chunk-relative symbol positions
// exc (ascending), sym0 = offsets[q0].  Unsorted offsets are reported by the kernel; the clamp keeps q inside the chunk.
inline void exception_queries(const uint64_t *offsets, uint64_t fixed_len, uint64_t q0, uint64_t q1, uint64_t sym0,
                              const std::vector<uint64_t> &exc, std::vector<uint32_t> &out) {
    out.clear();
    for (uint64_t pos : exc) {
        const uint64_t q = offsets ? std::min(query_of_symbol(offsets, q0, q1 + 1, sym0 + pos) - q0, q1 - q0 - 1)
                                   : pos / fixed_len;
        if (out.empty() || out.back() != (uint32_t)q) out.push_back((uint32_t)q);
    }
}

struct Chunk {
    uint64_t q0, q1, sym0, sym1;
    bool pack;         // pack the chunk's IO bytes to 2 bits on the host
    bool bad_offsets;  // the offsets at its end decrease or leave the batch: query q0 is reported
    uint64_t cq() const { return q1 - q0; }
    uint64_t nsym() const { return sym1 - sym0; }
};

// The budget of link bytes per chunk doubles from `first` to `max` (fast pipeline fill, then few large launches) and the
// batch ends with a chunk of about `tail` (short drain).  A packed chunk holds four symbols per link byte.
// Hybrid (pinned IO bytes with the packer on): pinned bytes can also cross the link as they are, by DMA, without any CPU
// work, so the packer and the link share the batch.  Before the pool starts on a packed chunk (which keeps the CPU busy
// for t_pack), a raw chunk is put on the link that is just large enough to keep it busy for that long on top of what is
// still queued there.  The caller observes the queue and passes it to after_upload, so a wrong guess of either rate
// corrects itself: too much raw data -> the backlog grows -> the next raw chunks shrink.
struct ChunkPlan {
    const uint64_t *offsets;  // the batch: offsets (nq + 1), or fixed_len + first_symbol
    uint64_t fixed_len, first_symbol, nq;
    bool prepacked;  // the caller's symbols are 2-bit packed
    bool pack;       // pack IO bytes on the host
    bool hybrid;     // pinned IO bytes with the packer on
    uint64_t first, max, tail;  // link bytes: budget of the first chunk, largest budget, size of the last chunk
    uint64_t max_queries;
    double pack_rate;                  // of the host packer, symbols per ms: a first guess, refined from every packed chunk
    double link_bytes_per_ms = 50e6;  // a first guess of the host-to-device link rate (50 GB/s)
    uint64_t budget = first, raw_want = first, q0 = 0;
    bool raw_next = hybrid;  // the link is idle at the start: open with a raw chunk
    uint64_t sym(uint64_t q) const { return offsets ? offsets[q] : q * fixed_len + first_symbol; }
    // the largest number of symbols a chunk of more than one query can hold
    uint64_t max_chunk_symbols() const { return std::min<uint64_t>(sym(nq) - sym(0), 4 * max); }
    // the next chunk, false once the batch is done
    bool next(Chunk &c) {
        if (q0 >= nq) return false;
        const bool raw_turn = hybrid && pack && raw_next, pack_chunk = pack && !raw_turn;
        const uint64_t unit = (pack_chunk || prepacked) ? 4 : 1;
        const uint64_t remaining = sym(nq) - sym(q0);
        uint64_t want = raw_turn ? raw_want : budget * unit;
        if (remaining <= want) want = remaining > 2 * tail * unit ? remaining - tail * unit : remaining;
        uint64_t q1 = offsets ? std::max(query_of_symbol(offsets, q0 + 1, nq + 1, offsets[q0] + want), q0 + 1)
                              : q0 + (fixed_len ? std::max<uint64_t>(1, want / fixed_len) : max_queries);
        q1 = std::min<uint64_t>(q1, std::min<uint64_t>(nq, q0 + max_queries));
        if (pack_chunk || !(hybrid && pack)) budget = std::min<uint64_t>(budget * 2, max);
        // (inside a chunk the kernel checks every query)
        c = Chunk{q0, q1, sym(q0), sym(q1), pack_chunk, sym(q1) < sym(q0) || sym(q1) > sym(nq)};
        q0 = q1;
        return true;
    }
    // the batch is not one of plain searchable symbols: IO bytes from here on (the chunk already cut keeps its size)
    void packing_failed() { pack = false; }
    // hybrid: after the upload of a chunk (packed: host-packed, nsym symbols staged in stage_ms) with
    // link_backlog_bytes still queued on the link
    void after_upload(bool packed, uint64_t nsym, double stage_ms, uint64_t link_backlog_bytes) {
        if (!packed) {
            raw_next = false;  // a raw chunk is always followed by a packed one
            return;
        }
        if (stage_ms > 0.02) pack_rate = 0.5 * pack_rate + 0.5 * (double)nsym / stage_ms;
        // how long will the pool need for the next packed chunk, and will the link last that long?
        const double t_pack = (double)(budget * 4) / pack_rate;
        const double have = (double)link_backlog_bytes;
        const double need = t_pack * link_bytes_per_ms;
        raw_next = pack && need - have >= (double)(2ull << 20);
        raw_want = raw_next ? std::min<uint64_t>((uint64_t)(need - have), 4 * max) : 0;
    }
};

}  // namespace gdx
