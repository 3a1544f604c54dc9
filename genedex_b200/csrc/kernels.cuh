// kernels.cuh -- hand-written sm_100a kernels of the search path.
//
//   k_query_keys    sort key (last 12 symbols) of every query; cub radix sort then gives the order in
//                   which threads pick queries, so that the top of the search trie is shared in L2
//   k_search        K1+K2: lookup-table seed + backward search, one thread per query, both interval
//                   borders' records in flight together      (batch_computed_cursors.rs:36-172,
//                                                              lookup_table.rs:68-161, condensed.rs:137-341)
//                   <.., VERIFY>: one-row intervals are finished by resolving SA[row] and comparing the
//                   rest of the query with the text section (count / locate only, identical results)
//   k_extend        one LF pair per cursor                   (cursor.rs:34-51)
//   k_hamming       backtracking backward search with up to k substitutions, one thread per query (hamming.h;
//                   no counterpart in the reference)
//   k_interval_counts / k_expand_rows / k_expand_big_rows / k_add_base    rows of every hit (CSR)
//   k_locate_walk   K3+K4: LF-walk to the next SA sample + text-id mapping, one thread per hit
//                                                             (sampled_suffix_array.rs:110-138,
//                                                              text_id_search_tree.rs:35-64)
//   k_pack_*        BWT -> rank records (+ per-superblock totals)        (condensed.rs:59-124,365-415)
//   k_pack_text     dense text -> 4/8-bit text section
//   k_lut_fill      lookup level d from level d-1            (lookup_table.rs:163-258)
//   k_ref_blocks_to_bwt  the reference's block arrays (condensed / flat, Block64 / Block512) -> dense BWT
//   k_records_to_bwt device records -> dense BWT (export)
//   k_densify       SA[row] for every row from the sampled suffix array (accelerator)
//   k_build_row_context  SA[row] + 45 symbols of text context per row (accelerator)
//   k_lut_extend    one level of the seed table (accelerator: a deeper lookup level outside the image)
//   k_gather        random-gather ceiling microbenchmark     (SURVEY 8d)
//
// All hot loads are random sector accesses into HBM: there is no reuse to stage through shared
// memory or TMA, so the design levers are (1) one aligned record per rank, fetched with a single
// 256-bit LDG.NA (no L1 allocation, keeps L1 for the superblock table and the text comparison),
// (2) both borders issued back to back, one fetch when they share a block, (3) enough resident warps
// to keep the DRAM random-access rate saturated, (4) fewer random fetches per query: suffix-sorted
// query order (L2 serves the first ~10 steps), text verification (~16 LF steps instead of 50, word-wise
// comparison) and the dense suffix array (SA[row] in one load), (5) few instructions per step: at 12 warps
// per scheduler an LF iteration takes about as long to issue as a DRAM round trip.  DRAM serves every
// random access as a whole 128 B line (profiles/r1_gather_dram.txt); a record is one 32 B sector of it.
#ifndef GDX_KERNELS_CUH
#define GDX_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>

#include <cub/block/block_scan.cuh>

#include "device_index.h"
#include "hamming.h"
#include "row_context.h"

namespace gdx {

struct DevQueries {
    const uint8_t *bytes;     // IO bytes, or nullptr when `packed` is set
    const uint64_t *offsets;  // nq + 1 entries or nullptr
    const uint32_t *offsets32;  // the same, chunk relative and narrow (host pipeline: half the PCIe bytes), or nullptr
    uint64_t fixed_len;
    uint64_t nq;
    uint64_t base;            // subtracted from offsets[] (chunked uploads)
    uint64_t shift;           // added to the start of every query (a packed chunk need not start on a byte boundary)
    // 2-bit packed form (alphabets with <= 4 searchable symbols): symbol i of the batch (the same index
    // that addresses `bytes`) sits at bits [2i, 2i+2) of this little-endian word stream, code = dense - 1.
    // The host packer routes queries with any other byte to the IO-byte kernel, so its batches hold searchable
    // symbols only.  A caller's pre-packed batch of an alphabet with fewer than 4 searchable symbols can hold
    // codes >= ns: k_search checks those queries in full before it searches them (packed_query_unsearchable).
    const uint32_t *packed;
    // number of symbols the stream holds (host pipeline: the chunk that was uploaded; ~0 = unknown): a query whose
    // offsets point outside is reported instead of read -- offsets are caller data and not checked on the host
    uint64_t limit;
};

// symbols [begin, begin + len) of the batch's stream belong to query q
__device__ __forceinline__ void query_extent(const DevQueries &qs, uint64_t q, uint64_t &begin, uint64_t &len) {
    if (qs.offsets32) {
        const uint32_t b = __ldg(qs.offsets32 + q);
        begin = b;
        len = __ldg(qs.offsets32 + q + 1) - b;
    } else if (qs.offsets) {
        begin = __ldg(qs.offsets + q) - qs.base;
        len = __ldg(qs.offsets + q + 1) - qs.base - begin;
    } else {
        begin = q * qs.fixed_len;
        len = qs.fixed_len;
    }
    begin += qs.shift;
}

// ---- 2-bit packed queries ----------------------------------------------------------------------------
// The last 64 symbols of a query live in two registers: symbol j (counted from the first staged symbol)
// at bits [2j, 2j+2) of the 128-bit value hi:lo.
// (struct PackedTail: row_context.h)
__device__ __forceinline__ uint32_t packed_code_global(const uint32_t *pk, uint64_t g) {
    return (__ldg(pk + (g >> 4)) >> ((uint32_t)(g & 15) * 2)) & 3u;
}
// symbols [g0, g0 + nsym) of the stream, nsym <= 64; words past the last needed one are not touched
__device__ __forceinline__ PackedTail load_packed_tail(const uint32_t *pk, uint64_t g0, uint32_t nsym) {
    const uint32_t *w = pk + (g0 >> 4);
    const uint32_t sh = (uint32_t)(g0 & 15) * 2;
    const uint32_t nw = ((uint32_t)(g0 & 15) + nsym + 15u) >> 4;  // <= 5
    uint32_t v[5];
#pragma unroll
    for (uint32_t k = 0; k < 5; ++k) v[k] = k < nw ? __ldg(w + k) : 0u;
    uint32_t t[4];
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k) t[k] = __funnelshift_r(v[k], v[k + 1], sh);
    PackedTail r;
    r.lo = (uint64_t)t[0] | ((uint64_t)t[1] << 32);
    r.hi = (uint64_t)t[2] | ((uint64_t)t[3] << 32);
    return r;
}
// 2 * nsym bits starting at staged symbol `sym` (nsym <= 32; bits past symbol 63 read as 0)
__device__ __forceinline__ uint64_t tail_bits(const PackedTail &t, uint32_t sym, uint32_t nsym) {
    const uint32_t bit = sym * 2;
    uint64_t v;
    if (bit == 0) v = t.lo;
    else if (bit < 64) v = (t.lo >> bit) | (t.hi << (64 - bit));
    else v = bit < 128 ? t.hi >> (bit - 64) : 0ull;
    return nsym >= 32 ? v : v & ((1ull << (2 * nsym)) - 1ull);
}
__device__ __forceinline__ uint32_t tail_code(const PackedTail &t, uint32_t sym) {
    return (uint32_t)((sym < 32 ? t.lo : t.hi) >> ((sym & 31u) * 2)) & 3u;
}
// true if a symbol of the packed query [begin, begin + tail_begin + tail) is not searchable; `t` holds its last `tail`
// symbols.  Looks at the whole query, whatever part of it the search would reach.
__device__ __noinline__ bool packed_query_unsearchable(const uint32_t *pk, uint64_t begin, uint64_t tail_begin,
                                                       PackedTail t, uint32_t tail, uint32_t ns) {
    if (packed_codes_unsearchable(t, tail, ns)) return true;
    for (uint64_t j0 = 0; j0 < tail_begin; j0 += 64) {
        const uint32_t nsym = tail_begin - j0 < 64 ? (uint32_t)(tail_begin - j0) : 64u;
        if (packed_codes_unsearchable(load_packed_tail(pk, begin + j0, nsym), nsym, ns)) return true;
    }
    return false;
}
// 16 2-bit codes -> 16 nibbles holding dense symbols (code + 1); 8 codes -> 8 bytes
__device__ __forceinline__ uint64_t expand_codes_4(uint64_t x) {
    x &= 0xffffffffull;
    x = (x | (x << 16)) & 0x0000ffff0000ffffull;
    x = (x | (x << 8)) & 0x00ff00ff00ff00ffull;
    x = (x | (x << 4)) & 0x0f0f0f0f0f0f0f0full;
    x = (x | (x << 2)) & 0x3333333333333333ull;
    return x + 0x1111111111111111ull;
}
__device__ __forceinline__ uint64_t expand_codes_8(uint64_t x) {
    x &= 0xffffull;
    x = (x | (x << 24)) & 0x000000ff000000ffull;
    x = (x | (x << 12)) & 0x000f000f000f000full;
    x = (x | (x << 6)) & 0x0303030303030303ull;
    return x + 0x0101010101010101ull;
}

constexpr uint64_t kNoError = ~0ull;

// ---- loads -------------------------------------------------------------------------------------
__device__ __forceinline__ void ldg256_na(const void *p, uint64_t w[4]) {
    asm("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
        : "=l"(w[0]), "=l"(w[1]), "=l"(w[2]), "=l"(w[3])
        : "l"(p));
}
__device__ __forceinline__ void ldg128_na(const void *p, uint64_t &lo, uint64_t &hi) {
    asm("ld.global.nc.L1::no_allocate.v2.u64 {%0,%1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(p));
}

// ---- layout traits -----------------------------------------------------------------------------
struct K32 {
    static constexpr uint32_t kLog2P = 6;
    static constexpr int kSearchMinBlocks = 6;  // 40 registers: 1536 threads per SM
    static constexpr int kVerifyMinBlocks = 6;
    struct Planes {
        uint64_t w[4];
    };
    struct Rec {
        uint64_t w[4];
    };
    static __device__ __forceinline__ Planes load_planes(const DevIndex &ix, uint64_t i) {
        Planes r;
        ldg256_na(ix.records + ((i >> 6) << 5), r.w);
        return r;
    }
    static __device__ __forceinline__ Rec load(const DevIndex &ix, uint64_t i, uint32_t) {
        Rec r;
        ldg256_na(ix.records + ((i >> 6) << 5), r.w);
        return r;
    }
    // a record that will not be needed again (one-row interval, locate walk).  An L2 evict_first policy on
    // these loads was measured: no effect on B200 (profiles/README.md), so they are plain loads.
    static __device__ __forceinline__ Rec load_once(const DevIndex &ix, uint64_t i, uint32_t) {
        Rec r;
        ldg256_na(ix.records + ((i >> 6) << 5), r.w);
        return r;
    }
    static __device__ __forceinline__ Planes load_planes_once(const DevIndex &ix, uint64_t i) {
        Planes r;
        ldg256_na(ix.records + ((i >> 6) << 5), r.w);
        return r;
    }
    static __device__ __forceinline__ Rec with_offset(const DevIndex &, const Planes &p, uint64_t,
                                                      uint32_t) {
        Rec r;
#pragma unroll
        for (int k = 0; k < 4; ++k) r.w[k] = p.w[k];
        return r;
    }
    static __device__ __forceinline__ uint32_t symbol_at(const Planes &p, uint64_t i) {
        return k32_symbol_at(p.w, (uint32_t)(i & 63));
    }
    static __device__ __forceinline__ uint32_t local_rank(const Rec &r, uint32_t c, uint64_t i) {
        return k32_local_rank(r.w, c, (uint32_t)(i & 63));
    }
    // LF of the symbol without an in-record offset (sigma == 6: dense 5 = `N`), see rank_core.h
    static __device__ __noinline__ uint64_t lf_derived(const DevIndex &ix, uint64_t i) {
        uint64_t w[4];
        ldg256_na(ix.records + ((i >> 6) << 5), w);
        uint64_t others = k32_local_rank_sum(w, (uint32_t)(i & 63));
        const uint64_t *sb = ix.sbc + (i >> kSuperblockLog2) * 4;
#pragma unroll
        for (uint32_t c = 1; c <= 4; ++c) others += __ldg(sb + (c - 1)) - __ldg(ix.count + c);
        uint64_t rank0 = lower_bound_u64(ix.border_rows, ix.n_border, i);
        return __ldg(ix.count + 5) + (i - rank0 - others);
    }
};

template <int B>
struct KG {
    static constexpr uint32_t kLog2P = 7;
    static constexpr int kPlanes = B;
    static constexpr int kSearchMinBlocks = B <= 3 ? 5 : (B <= 5 ? 5 : 3);
    static constexpr int kVerifyMinBlocks = B <= 5 ? 5 : 3;
    // The record is fetched as whole 32 B sectors: kSectors 256-bit loads cover the B planes (16 B each) and the
    // first u16 offsets behind them; an offset further back costs one more 2-byte load from the same line.
    // (Protein, B = 5: 3 sector requests instead of five 128-bit ones + the offset -- the random-access ceiling
    // of the part counts sector requests, profiles/r1_gather_ceiling.json.)
    static constexpr int kSectors = (16 * B + 31) / 32;
    static constexpr int kWords = 4 * kSectors;           // u64 words held in registers
    static constexpr uint32_t kOffsetsInRegs = (32 * kSectors - 16 * B) / 2;  // offsets of symbols 1..this many
    struct Planes {
        uint64_t w[kWords];
    };
    struct Rec {
        uint64_t w[kWords];
        uint32_t off;
    };
    static __device__ __forceinline__ const uint8_t *rec_ptr(const DevIndex &ix, uint64_t i) {
        return ix.records + (i >> 7) * ix.stride;
    }
    static __device__ __forceinline__ void load_words(const uint8_t *p, uint64_t *w) {
#pragma unroll
        for (int k = 0; k < kSectors; ++k) ldg256_na(p + 32 * k, w + 4 * k);
    }
    static __device__ __forceinline__ uint32_t offset_of(const uint8_t *p, const uint64_t *w, uint32_t c) {
        if (kOffsetsInRegs > 0 && c <= kOffsetsInRegs) {
            uint32_t v = 0;  // compile-time word indices only: a run-time index would push the record to local memory
#pragma unroll
            for (uint32_t j = 0; j < kOffsetsInRegs; ++j) {
                const uint32_t byte = 16 * B + 2 * j;  // position of the offset inside the loaded sectors
                if (c - 1 == j) v = (uint32_t)(w[byte >> 3] >> ((byte & 7) * 8)) & 0xffffu;
            }
            return v;
        }
        return __ldg(reinterpret_cast<const uint16_t *>(p + 16 * B) + (c - 1));
    }
    static __device__ __forceinline__ Planes load_planes(const DevIndex &ix, uint64_t i) {
        Planes r;
        load_words(rec_ptr(ix, i), r.w);
        return r;
    }
    static __device__ __forceinline__ Rec load(const DevIndex &ix, uint64_t i, uint32_t c) {
        Rec r;
        const uint8_t *p = rec_ptr(ix, i);
        load_words(p, r.w);
        r.off = offset_of(p, r.w, c);
        return r;
    }
    static __device__ __forceinline__ Rec load_once(const DevIndex &ix, uint64_t i, uint32_t c) { return load(ix, i, c); }
    static __device__ __forceinline__ Planes load_planes_once(const DevIndex &ix, uint64_t i) { return load_planes(ix, i); }
    static __device__ __forceinline__ Rec with_offset(const DevIndex &ix, const Planes &pl, uint64_t i,
                                                      uint32_t c) {
        Rec r;
#pragma unroll
        for (int k = 0; k < kWords; ++k) r.w[k] = pl.w[k];
        r.off = offset_of(rec_ptr(ix, i), pl.w, c);
        return r;
    }
    // plane p = words 2p (positions 0..63) and 2p + 1 (64..127)
    static __device__ __forceinline__ uint32_t symbol_at(const Planes &p, uint64_t i) {
        const uint32_t bit = (uint32_t)(i & 127), sh = bit & 63u, hi = bit >> 6;
        uint32_t s = 0;
#pragma unroll
        for (int k = 0; k < B; ++k) s |= (uint32_t)(((hi ? p.w[2 * k + 1] : p.w[2 * k]) >> sh) & 1u) << k;
        return s;
    }
    static __device__ __forceinline__ uint32_t local_rank(const Rec &r, uint32_t c, uint64_t i) {
        const uint32_t bit = (uint32_t)(i & 127);
        uint64_t mlo = ~0ull, mhi = ~0ull;
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const bool one = (c >> k) & 1u;
            mlo &= one ? r.w[2 * k] : ~r.w[2 * k];
            mhi &= one ? r.w[2 * k + 1] : ~r.w[2 * k + 1];
        }
        const uint64_t masklo = below(bit), maskhi = bit > 64 ? below(bit - 64) : 0ull;
        return r.off + (uint32_t)(popc64(mlo & masklo) + popc64(mhi & maskhi));
    }
    static __device__ __forceinline__ uint64_t lf_derived(const DevIndex &, uint64_t i) { return i; }
};

__device__ __forceinline__ uint64_t sbc_load(const DevIndex &ix, uint64_t i, uint32_t c) {
    return __ldg(ix.sbc + (i >> kSuperblockLog2) * ix.noff + (c - 1));
}

// LF(c, s), LF(c, e) with all loads issued before the first use (lib.rs:273-275).  Once the interval
// is narrower than a block both borders usually live in the same record: it is fetched once.
template <class L>
__device__ __forceinline__ void lf_pair(const DevIndex &ix, uint32_t c, uint64_t &s, uint64_t &e) {
    if (c > ix.noff) {  // derived symbol: rare and divergent by nature
        s = L::lf_derived(ix, s);
        e = L::lf_derived(ix, e);
        return;
    }
    const bool same_block = (s >> L::kLog2P) == (e >> L::kLog2P);
    // narrow intervals are private to this query: their records are streamed through L2 (evict first)
    typename L::Rec rs = (same_block && e - s <= 2) ? L::load_once(ix, s, c) : L::load(ix, s, c);
    const uint64_t bs = sbc_load(ix, s, c);
    if (same_block) {
        const uint64_t ns = bs + L::local_rank(rs, c, s);
        e = bs + L::local_rank(rs, c, e);
        s = ns;
        return;
    }
    typename L::Rec re = L::load(ix, e, c);
    const uint64_t be = sbc_load(ix, e, c);
    s = bs + L::local_rank(rs, c, s);
    e = be + L::local_rank(re, c, e);
}

__device__ __forceinline__ void lut_load(const DevIndex &ix, uint64_t entry, uint64_t &s, uint64_t &e) {
    if (ix.wide) {
        ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(ix.lookup) + entry);
        s = v.x;
        e = v.y;
    } else {
        uint2 v = __ldg(reinterpret_cast<const uint2 *>(ix.lookup) + entry);
        s = v.x;
        e = v.y;
    }
}

__device__ __forceinline__ void seed_load(const DevIndex &ix, uint64_t entry, uint64_t &s, uint64_t &e) {
    if (ix.wide) {
        const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(ix.seed_lookup) + entry);
        s = v.x;
        e = v.y;
    } else {
        const uint2 v = __ldg(reinterpret_cast<const uint2 *>(ix.seed_lookup) + entry);
        s = v.x;
        e = v.y;
    }
}

__device__ __forceinline__ void report_error(uint64_t *err, uint64_t q) {
    if (err) atomicMin(reinterpret_cast<unsigned long long *>(err), (unsigned long long)q);
}

// ---- SA[row] by LF-walk to the next sample (sampled_suffix_array.rs:110-138) -------------------------
template <class L>
__device__ __forceinline__ uint64_t resolve_row(const DevIndex &ix, uint64_t i, uint32_t &steps) {
    for (;;) {
        const bool sampled = ix.sampling_shift != 0xffffffffu ? (i & ((1ull << ix.sampling_shift) - 1)) == 0
                                                              : (i % ix.sampling_rate) == 0;
        if (sampled) {
            const uint64_t k = ix.sampling_shift != 0xffffffffu ? i >> ix.sampling_shift : i / ix.sampling_rate;
            if (ix.wide) return __ldg(reinterpret_cast<const uint64_t *>(ix.samples) + k) + steps;
            const uint32_t *sp = reinterpret_cast<const uint32_t *>(ix.samples) + k;
            return (uint64_t)__ldg(sp) + steps;
        }
        typename L::Planes pl = L::load_planes_once(ix, i);
        const uint32_t c = L::symbol_at(pl, i);
        if (c == 0) {  // :121-126 text_border_lookup[&i]
            const uint64_t k = lower_bound_u64(ix.border_rows, ix.n_border, i);
            return __ldg(ix.border_pos + k) + steps;
        }
        if (c > ix.noff) {
            i = L::lf_derived(ix, i);
        } else {
            typename L::Rec r = L::with_offset(ix, pl, i, c);
            i = sbc_load(ix, i, c) + L::local_rank(r, c, i);
        }
        ++steps;
    }
}

// one LF step from an SA row: row of the suffix that starts one text position earlier (the BWT symbol of
// the row must not be the sentinel -- callers stay inside a region that matched query symbols)
template <class L>
__device__ __forceinline__ uint64_t lf_row(const DevIndex &ix, uint64_t row) {
    typename L::Planes pl = L::load_planes_once(ix, row);
    const uint32_t c = L::symbol_at(pl, row);
    if (c == 0) return row;
    if (c > ix.noff) return L::lf_derived(ix, row);
    typename L::Rec r = L::with_offset(ix, pl, row, c);
    return sbc_load(ix, row, c) + L::local_rank(r, c, row);
}

template <class L>
__device__ __forceinline__ uint64_t lf_one(const DevIndex &ix, uint32_t c, uint64_t i) {
    if (c > ix.noff) return L::lf_derived(ix, i);
    typename L::Rec r = L::load_once(ix, i, c);
    return sbc_load(ix, i, c) + L::local_rank(r, c, i);
}

// ISA[t] = SA row of the suffix starting at text position t, from the sampled inverse suffix array:
// start at the next sampled position q >= t and walk q - t LF steps back.  Every text position in [t, q)
// must hold a non-sentinel symbol (callers guarantee q lies inside a matched region).
template <class L>
__device__ __forceinline__ uint64_t isa_row(const DevIndex &ix, uint64_t t, uint32_t &steps) {
    const uint64_t k = (t + ix.isa_rate - 1) / ix.isa_rate;
    uint64_t row = ix.wide ? __ldg(reinterpret_cast<const uint64_t *>(ix.isa) + k)
                           : (uint64_t)__ldg(reinterpret_cast<const uint32_t *>(ix.isa) + k);
    for (uint64_t q = k * ix.isa_rate; q > t; --q) {
        row = lf_row<L>(ix, row);
        ++steps;
    }
    return row;
}

// dense symbol at concatenated-text position p (text section of the image)
__device__ __forceinline__ uint32_t text_symbol(const DevIndex &ix, uint64_t p) {
    if (ix.text_bits == 4) return (__ldg(ix.text + (p >> 1)) >> ((p & 1) * 4)) & 15u;
    return __ldg(ix.text + p);  // L1-allocating on purpose: the comparison walks consecutive bytes
}

// Right-to-left comparison of query[0..pos) with the text in front of position `at` (query position j
// <-> text position at - (pos - j)), a 64-bit word of packed symbols at a time.  Same outcome as the
// reference's one-rank-per-symbol shrinking of a one-row interval (cursor.rs:40-51):
//   0 = every symbol matched; 1 = first mismatch from the right at query position jm (symbol cm);
//   2 = an invalid symbol (dense 0, alphabet.rs:195-198) is reached before any mismatch.
// Positions before the start of the first text read as 0 = sentinel, which no valid symbol matches.
// The text section is padded so that the word after the last one may be read.
// query_word(j0, cnt): dense symbols of query positions [j0, j0 + cnt), BITS bits each, symbol j0 lowest.
// CHECK_ZERO = false: the query cannot hold an invalid symbol (2-bit packed batches).
template <int BITS, bool CHECK_ZERO, class QW>
__device__ __forceinline__ int compare_with_text(const DevIndex &ix, QW &&query_word, uint64_t pos, uint64_t at,
                                                 uint64_t &jm, uint32_t &cm) {
    constexpr uint32_t SPW = 64 / BITS;  // symbols per word
    constexpr uint64_t kLow = BITS == 4 ? 0x7777777777777777ull : 0x7f7f7f7f7f7f7f7full;
    const uint64_t *text64 = reinterpret_cast<const uint64_t *>(ix.text);
    uint64_t j_hi = pos;
    while (j_hi > 0) {
        const uint32_t cnt = j_hi < SPW ? (uint32_t)j_hi : SPW;
        const uint64_t j0 = j_hi - cnt;
        const uint64_t back0 = pos - j0;  // distance of query position j0 from `at`
        uint64_t tw;
        if (back0 <= at) {
            const uint64_t t0 = at - back0;
            const uint32_t sh = (uint32_t)(t0 % SPW) * BITS;
            const uint64_t w0 = __ldg(text64 + t0 / SPW), w1 = __ldg(text64 + t0 / SPW + 1);
            tw = sh ? (w0 >> sh) | (w1 << (64 - sh)) : w0;
        } else {  // the chunk starts before position 0 of the first text
            const uint64_t missing = back0 - at;
            tw = missing >= SPW ? 0 : __ldg(text64) << (missing * BITS);
        }
        const uint64_t qw = query_word(j0, cnt);
        const uint64_t vm = cnt == SPW ? ~0ull : (1ull << (cnt * BITS)) - 1;
        const uint64_t diff = (qw ^ tw) & vm;
        const uint64_t zero = CHECK_ZERO ? ~(((qw & kLow) + kLow) | qw | kLow) & vm : 0ull;  // top bit of every symbol that is 0
        if (diff | zero) {
            const uint32_t km = diff ? (63u - (uint32_t)__clzll((long long)diff)) / BITS : 0;
            if (CHECK_ZERO && zero && (!diff || (63u - (uint32_t)__clzll((long long)zero)) / BITS >= km)) return 2;
            jm = j0 + km;
            cm = (uint32_t)(qw >> (km * BITS)) & ((1u << BITS) - 1);
            return 1;
        }
        j_hi = j0;
    }
    return 0;
}

// ---- row context table (accelerator, gdx_index_set_row_context_table): layout and arithmetic in row_context.h ----

// query words of an IO-byte query whose last bytes are staged in shared memory (tab = io -> dense)
template <int BITS>
struct ByteQueryWords {
    const uint8_t *tab, *sbytes, *p;
    uint64_t tail_begin;
    __device__ __forceinline__ uint64_t operator()(uint64_t j0, uint32_t cnt) const {
        constexpr uint32_t SPW = 64 / BITS;
        uint64_t qw = 0;
        if (j0 >= tail_begin) {  // the whole chunk is staged: two 32-bit halves, no per-symbol branch
            const uint8_t *sp = sbytes + (j0 - tail_begin);
            uint32_t lo = 0, hi = 0;
#pragma unroll
            for (uint32_t k = 0; k < SPW / 2; ++k) {
                if (k < cnt) lo |= (uint32_t)tab[sp[k]] << (k * BITS);
                if (k + SPW / 2 < cnt) hi |= (uint32_t)tab[sp[k + SPW / 2]] << (k * BITS);
            }
            qw = (uint64_t)lo | ((uint64_t)hi << 32);
        } else {  // reaches in front of the staged tail of a long query
#pragma unroll 1
            for (uint32_t k = 0; k < cnt; ++k) {
                const uint64_t i = j0 + k;
                const uint32_t c = tab[i >= tail_begin ? sbytes[i - tail_begin] : __ldg(p + i)];
                qw |= (uint64_t)c << (k * BITS);
            }
        }
        return qw;
    }
};

// query words of a 2-bit packed query whose last 64 symbols are in registers
template <int BITS>
struct PackedQueryWords {
    PackedTail tail;
    const uint32_t *pk;
    uint64_t begin, tail_begin;  // stream index of query symbol 0; query position of the first staged symbol
    __device__ __forceinline__ uint64_t operator()(uint64_t j0, uint32_t cnt) const {
        constexpr uint32_t SPW = 64 / BITS;
        uint64_t codes;
        if (j0 >= tail_begin) {
            codes = tail_bits(tail, (uint32_t)(j0 - tail_begin), SPW);
        } else {
            codes = 0;
#pragma unroll 1
            for (uint32_t k = 0; k < cnt; ++k) {
                const uint64_t i = j0 + k;
                const uint32_t c = i >= tail_begin ? tail_code(tail, (uint32_t)(i - tail_begin))
                                                   : packed_code_global(pk, begin + i);
                codes |= (uint64_t)c << (2 * k);
            }
        }
        const uint64_t qw = BITS == 4 ? expand_codes_4(codes) : expand_codes_8(codes);
        return cnt == SPW ? qw : qw & ((1ull << (cnt * BITS)) - 1);
    }
};

// interval flag of the locate plumbing: start = resolved text position, end = kDirectHit
constexpr uint64_t kDirectHit = ~0ull;
// k_search switches from LF steps to "resolve the row + compare against the text" when the interval has
// one row and at least DevIndex::verify_min_remaining symbols are left (a walk + sample + text read costs
// about 5 random sectors; default 8, 4 once the dense suffix array is built; GDX_VERIFY_MIN overrides it for measurements)

// ---- sort key of a query: its last symbols, last symbol most significant ---------------------------
// Backward search consumes a query right to left, so queries that share a suffix walk the same
// records for their first steps.  Sorting the batch by suffix makes neighbouring threads/CTAs walk
// them at the same time: the top of the search trie is then served by L2 instead of DRAM (the
// north-star "query batches are sorted by lookup-table prefix so they share L2").  The sort only
// permutes the order in which threads pick queries; every result still goes to the query's own slot.
// sort key of query q: its last key_syms symbols, the last symbol most significant (unsearchable / invalid
// symbols and positions in front of a short query count as code 0)
__device__ __forceinline__ uint32_t query_sort_key(const DevIndex &ix, const DevQueries &qs, uint64_t q,
                                                   uint32_t key_bits, uint32_t key_syms) {
    uint64_t begin, len;
    query_extent(qs, q, begin, len);
    uint32_t key = 0;
    for (uint32_t j = 0; j < key_syms; ++j) {
        uint32_t code = 0;
        if (j < len) {
            if (qs.packed) {
                code = packed_code_global(qs.packed, begin + len - 1 - j);
            } else {
                const uint32_t c = ix.io_to_dense[__ldg(qs.bytes + begin + len - 1 - j)];
                code = (c >= 1 && c <= ix.ns) ? c - 1 : 0;
            }
        }
        key = (key << key_bits) | code;
    }
    return key;
}

__global__ void __launch_bounds__(256)
k_query_keys(const __grid_constant__ DevIndex ix, const DevQueries qs, uint32_t key_bits, uint32_t key_syms,
             uint32_t *__restrict__ keys, uint32_t *__restrict__ idx) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= qs.nq) return;
    keys[q] = query_sort_key(ix, qs, q, key_bits, key_syms);
    idx[q] = (uint32_t)q;
}

// ---- K1 + K2: seed + backward search ----------------------------------------------------------------
// mode 0: out_a = starts, out_b = ends; mode 1: out_a = counts.
// Follows the batched path of the reference: a symbol is translated only when the search reaches
// it (batch_computed_cursors.rs:84-87,106-113), queries leave when all symbols are consumed or the
// interval is empty (:131-158), results are written to the query's own slot (= input order, :160-172).
// perm (optional): thread t searches query perm[t] (suffix-sorted order, see k_query_keys).
// The last kQueryStage bytes of the query are staged once into a private shared-memory slot with
// aligned word loads; the per-step symbol fetch is then an LDS, not a global byte load.
constexpr uint32_t kQueryStage = 64;                       // bytes staged per query
constexpr uint32_t kQuerySlotWords = kQueryStage / 4 + 1;  // 17: odd stride, covers any misalignment

// VERIFY (count / locate only, needs the text section): as soon as the interval holds exactly one row
// and >= verify_min_remaining symbols are left, SA[row] is resolved (LF-walk to a sample) and the rest
// of the query is compared with the text right to left.  The reference would shrink that interval to
// [x, x+1) or to empty by the same comparisons, one rank per symbol (cursor.rs:40-51): count and hit
// are identical, the invalid-symbol panic fires at the same symbol, only the interval itself is not
// produced -- so mode 0 (cursors) never uses it.  mode 2 = locate: out_a/out_b carry either the
// interval or (text position, kDirectHit).
// CURSORS (mode 0 with VERIFY): compile the inverse-sample path only into the variant that needs it
// PACKED: the batch is a 2-bit packed stream (DevQueries::packed); the last 64 symbols of a query are held
// in two registers (no shared-memory staging, no translate table), lookup indices are bit-field extracts
// when ns == 4, and the only invalid symbols are codes >= ns (ns < 4), refused before the search starts.
// slot_map (optional): the result of query q goes to slot slot_map[q] (queries re-run through the IO-byte
// kernel because they hold a byte the packer cannot encode); errors are reported for that slot.
// out_bits: 64 or 32 (narrow results for texts shorter than 2^32: half the D2H bytes).
constexpr int kModeNarrow = 8;  // mode flag: results are written as uint32
// error word of k_search: smallest failing query index (atomicMin); a query whose offsets leave the uploaded stream
// carries this flag (so an invalid symbol in an earlier or later query still wins the report, as it would in the
// reference, which cannot express broken offsets at all)
constexpr uint64_t kBadOffsetFlag = 1ull << 62;

// what k_search adds up over its queries (warp totals, atomicAdd)
struct SearchCounters {
    unsigned long long lf_steps;           // LF steps of the search
    unsigned long long verify_walk_steps;  // walk steps of the rows verified through the text section
    unsigned long long verified_rows;      // rows verified through the text section
};

template <class L, bool VERIFY, bool CURSORS, bool PACKED>
__global__ void __launch_bounds__(256, VERIFY ? L::kVerifyMinBlocks : L::kSearchMinBlocks)
k_search(const __grid_constant__ DevIndex ix, const DevQueries qs, uint64_t *__restrict__ out_a,
         uint64_t *__restrict__ out_b, int mode_flags, uint64_t q_index_base, uint64_t *err,
         SearchCounters *stats, const uint32_t *__restrict__ perm,
         const uint32_t *__restrict__ slot_map) {
    constexpr uint32_t kTabBytes = PACKED ? 4 : 256;
    constexpr uint32_t kStageWords = PACKED ? 1 : 256 * kQuerySlotWords;
    __shared__ uint8_t tab[kTabBytes];
    __shared__ uint16_t tab2[PACKED ? 2 : 256];  // io byte -> 2-bit code | 0x100 (codes_from_staged), ns <= 4 only
    __shared__ uint32_t stage[kStageWords];
    if constexpr (!PACKED) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) {
            const uint32_t d = ix.io_to_dense[i];
            tab[i] = (uint8_t)d;
            tab2[i] = ctx_tab2_entry(d, ix.ns);
        }
        __syncthreads();
    }
    const int mode = mode_flags & 7;
    const bool narrow = (mode_flags & kModeNarrow) != 0;

    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t steps = 0, vsteps = 0, vrows = 0;
    if (t < qs.nq) {
        const uint64_t q = perm ? (uint64_t)__ldg(perm + t) : t;
        uint64_t begin, len;
        query_extent(qs, q, begin, len);
        // decreasing / out-of-range offsets: nothing of the query is read, its result is the empty interval
        const bool broken = (qs.offsets32 || qs.offsets) && (begin > qs.limit || len > qs.limit - begin);
        if (broken) len = 0;
        const uint8_t *p = PACKED ? nullptr : qs.bytes + begin;

        // the last kQueryStage symbols of the query
        const uint32_t tail = len < kQueryStage ? (uint32_t)len : kQueryStage;
        const uint64_t tail_begin = len - tail;  // query position of the first staged symbol
        PackedTail ptail = {0, 0};
        const uint8_t *sbytes = nullptr;
        bool coded = PACKED;  // the staged symbols are held as 2-bit codes in ptail
        bool bad = false;
        if constexpr (PACKED) {
            if (tail) ptail = load_packed_tail(qs.packed, begin + tail_begin, tail);
            // With fewer than 4 searchable symbols a caller's pre-packed batch can hold a code that is none: it would
            // index the lookup / seed tables and the rank tables out of range.  Refused as an invalid symbol, whether or
            // not the search would reach it (a packed batch has no lazy reference behaviour to keep).
            if (ix.ns < 4 && tail) bad = packed_query_unsearchable(qs.packed, begin, tail_begin, ptail, tail, ix.ns);
        } else {
            // aligned words covering bytes [len - tail, len), global -> shared without a register round
            // trip: all words of the query are in flight at once
            uint32_t *slot = stage + threadIdx.x * kQuerySlotWords;
            const uint8_t *first = p + tail_begin;
            const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(first) & 3u);
            if (tail) {
                const uint32_t *w = reinterpret_cast<const uint32_t *>(first - mis);
                const uint32_t nw = (mis + tail + 3u) >> 2;
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(slot);
#pragma unroll 1
                for (uint32_t k = 0; k < nw; ++k)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4 * k), "l"(w + k) : "memory");
                asm volatile("cp.async.wait_all;" ::: "memory");
            }
            sbytes = reinterpret_cast<const uint8_t *>(slot) + mis;
            // (pays with the row context table, where the kernel is bound by instructions; without the table it is
            // bound by DRAM round trips and this pass in front of the first dependent load costs 5 % -- 6.50 -> 6.83
            // ms per 60 M queries -- but making it conditional on the table costs the common case registers)
            // The kernels without text verification run every LF step and are bound by rank records: left as they were.
            if constexpr (VERIFY) {
                if (ix.ns <= 4 && tail) coded = codes_from_staged(tab2, slot, mis, tail, ptail);
            }
        }
        // dense symbol of query position i
        auto symbol_at = [&](uint64_t i) -> uint32_t {
            if constexpr (PACKED)
                return 1u + (i >= tail_begin ? tail_code(ptail, (uint32_t)(i - tail_begin))
                                             : packed_code_global(qs.packed, begin + i));
            else if (i >= tail_begin)
                return coded ? 1u + tail_code(ptail, (uint32_t)(i - tail_begin)) : (uint32_t)tab[sbytes[i - tail_begin]];
            else
                return tab[__ldg(p + i)];
        };
        // lookup index of the d symbols starting at query position p0 (lookup_table.rs:68-161: the first
        // symbol is the least significant digit); ok = false if one of them is invalid or not searchable
        auto lookup_index = [&](uint64_t p0, uint32_t d, bool &ok) -> uint64_t {
            if (coded && ix.ns == 4 && d <= 32 && p0 >= tail_begin)  // the digits are the packed bits themselves
                return d ? tail_bits(ptail, (uint32_t)(p0 - tail_begin), d) : 0ull;
            uint64_t li = 0, f = 1;
            for (uint32_t j = 0; j < d; ++j) {
                const uint32_t c = symbol_at(p0 + j);
                if (c == 0 || c > ix.ns) ok = false;
                li += (uint64_t)(c - 1) * f;
                f *= ix.ns;
            }
            return li;
        };

        // K1: lookup_table.rs:68-161
        const uint32_t depth = len < ix.lookup_depth ? (uint32_t)len : ix.lookup_depth;
        uint64_t pos = len - depth;
        uint64_t s = 0, e = 0;
        // Seed table accelerator (gdx_index_set_seed_table_depth): one level of a lookup table deeper than
        // the configured one.  Its entries are exactly what the configured table + LF steps produce (an empty
        // interval stays as it was when it became empty, k_lut_extend), so it may stand in whenever all of its
        // symbols are searchable; anything else (invalid byte, `N`, short query) takes the configured path,
        // which keeps the reference's lazy panic and the documented deviation where they were.
        bool seeded = false;
        if (!bad && ix.seed_lookup && len >= ix.seed_depth) {
            const uint64_t p0 = len - ix.seed_depth;
            bool ok = true;
            const uint64_t li = lookup_index(p0, ix.seed_depth, ok);
            if (ok) {
                seed_load(ix, li, s, e);
                pos = p0;
                seeded = true;
            }
        }
        if (!seeded) {
            // c == 0: invalid symbol (alphabet.rs:195-198).  c > ns: valid but not searchable; the
            // reference mis-indexes its table here (lookup_table.rs:154-157) -- documented deviation.
            bool ok = true;
            const uint64_t li = lookup_index(pos, depth, ok);
            bad = bad || !ok || broken;
            if (!bad) lut_load(ix, ix.lut_level_off[depth] + li, s, e);
        }

        // K2: batch_computed_cursors.rs:62-70.  The verification runs inline, as soon as a lane's interval
        // has one row: its dependent DRAM fetches then overlap the LF steps of the other lanes of the warp
        // (deferring it behind the loop so that it runs once per warp was measured 22 % slower).
        bool direct = false;
        while (!bad && pos > 0 && s != e) {
            // mode 0 (cursors) must also produce the interval: possible with the sampled inverse suffix
            // array once at least sampling_rate symbols have matched (the ISA walk stays inside them)
            if (VERIFY && e - s == 1 && pos >= ix.verify_min_remaining &&
                (!CURSORS || len - pos >= ix.isa_rate)) {
                // one candidate row: SA[s] is where query[pos..len) occurs; compare query[0..pos)
                uint64_t at;
                vrows = 1;
                uint64_t jm = 0;     // query position of the first mismatch (from the right)
                uint32_t cm = 0;     // its dense symbol
                int cmp = -1;
                if (!CURSORS && ix.row_context) {
                    // count / locate with the row context table: position and context in one 16-byte load
                    CtxEntry en;
                    {
                        uint64_t e0, e1;
                        ldg128_na(reinterpret_cast<const uint4 *>(ix.row_context) + s, e0, e1);
                        en = CtxEntry{(uint32_t)e0, (uint32_t)(e0 >> 32), (uint32_t)e1, (uint32_t)(e1 >> 32)};
                    }
                    at = en.x;
                    if (coded && tail_begin == 0 && pos <= ctx_valid_len(en))
                        cmp = ctx_matches(en, (uint32_t)pos, ptail.lo, ptail.hi) ? 0 : 1;
                } else {
                    at = resolve_row<L>(ix, s, vsteps);
                }
                if (cmp >= 0) {
                    // decided from the entry (a mismatch needs no position: the interval is empty either way)
                } else if constexpr (PACKED) {
                    cmp = ix.text_bits == 4
                              ? compare_with_text<4, false>(ix, PackedQueryWords<4>{ptail, qs.packed, begin, tail_begin}, pos, at, jm, cm)
                              : compare_with_text<8, false>(ix, PackedQueryWords<8>{ptail, qs.packed, begin, tail_begin}, pos, at, jm, cm);
                } else {
                    cmp = ix.text_bits == 4
                              ? compare_with_text<4, true>(ix, ByteQueryWords<4>{tab, sbytes, p, tail_begin}, pos, at, jm, cm)
                              : compare_with_text<8, true>(ix, ByteQueryWords<8>{tab, sbytes, p, tail_begin}, pos, at, jm, cm);
                }
                const bool match = cmp == 0;
                bad = cmp == 2;  // the reference reaches this symbol with a non-empty interval
                if (bad) {
                    s = e = 0;
                } else if (!CURSORS) {
                    if (match) {
                        direct = true;
                        s = at - pos;  // text position of the whole query
                        e = s + 1;
                    } else {
                        s = e = 0;
                    }
                } else if (match) {
                    // the reference ends on [y, y + 1), y = row of the suffix at the query's text position
                    s = isa_row<L>(ix, at - pos, vsteps);
                    e = s + 1;
                } else {
                    // the reference's interval became empty at query[jm]: both borders of the one-row
                    // interval [r, r + 1) of query[jm+1..] map to count[c] + rank(c, r)  (lib.rs:273-275)
                    const uint64_t r = isa_row<L>(ix, at - (pos - jm - 1), vsteps);
                    s = e = lf_one<L>(ix, cm, r);
                }
                break;
            }
            const uint32_t c = symbol_at(pos - 1);
            if (!PACKED && c == 0) {
                bad = true;
                break;
            }
            lf_pair<L>(ix, c, s, e);
            --pos;
            ++steps;
        }
        const uint64_t slot_q = slot_map ? (uint64_t)__ldg(slot_map + q) : q;
        if (bad) {
            report_error(err, (broken ? kBadOffsetFlag : 0ull) | (q_index_base + slot_q));
            s = e = 0;
            direct = false;
        }
        if (narrow) {
            uint32_t *a32 = reinterpret_cast<uint32_t *>(out_a), *b32 = reinterpret_cast<uint32_t *>(out_b);
            if (mode == 0) {
                a32[slot_q] = (uint32_t)s;
                b32[slot_q] = (uint32_t)e;
            } else {
                a32[slot_q] = (uint32_t)(e - s);
            }
        } else if (mode == 0) {
            out_a[slot_q] = s;
            out_b[slot_q] = e;
        } else if (mode == 1) {
            out_a[slot_q] = e - s;
        } else {
            out_a[slot_q] = s;
            out_b[slot_q] = direct ? kDirectHit : e;
        }
    }
    if (stats) {
        uint32_t tot = __reduce_add_sync(0xffffffffu, steps);
        if ((threadIdx.x & 31) == 0 && tot) atomicAdd(&stats->lf_steps, (unsigned long long)tot);
        if (VERIFY) {
            tot = __reduce_add_sync(0xffffffffu, vsteps);
            if ((threadIdx.x & 31) == 0 && tot) atomicAdd(&stats->verify_walk_steps, (unsigned long long)tot);
            tot = __reduce_add_sync(0xffffffffu, vrows);
            if ((threadIdx.x & 31) == 0 && tot) atomicAdd(&stats->verified_rows, (unsigned long long)tot);
        }
    }
}

// ---- Cursor::extend_query_front for many cursors (cursor.rs:34-51) -----------------------------------
template <class L>
__global__ void __launch_bounds__(256)
k_extend(const __grid_constant__ DevIndex ix, uint64_t *__restrict__ starts, uint64_t *__restrict__ ends,
         const uint8_t *__restrict__ io_symbols, uint64_t n, uint64_t *err, uint64_t index_base) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    uint32_t c = ix.io_to_dense[io_symbols[q]];
    if (c == 0) {  // the reference translates before it looks at the interval (cursor.rs:35-37)
        report_error(err, index_base + q);
        return;
    }
    uint64_t s = starts[q], e = ends[q];
    if (s > ix.n || e > ix.n) {  // text_with_rank_support/mod.rs:106-110 bounds assert
        report_error(err + 1, index_base + q);
        return;
    }
    if (s != e) {
        lf_pair<L>(ix, c, s, e);
        starts[q] = s;
        ends[q] = e;
    }
}

// ---- Hamming search: rank sources of hamming_search (hamming.h) ---------------------------------------
// LF of the derived symbol (K32, sigma 6) from the sum of LF(c, i) over c = 1..4 (see K32::lf_derived)
__device__ __forceinline__ uint64_t k32_lf_derived_from_sum(const DevIndex &ix, uint64_t i, uint64_t lf_sum) {
    uint64_t counts = 0;
#pragma unroll
    for (uint32_t c = 1; c <= 4; ++c) counts += __ldg(ix.count + c);
    const uint64_t rank0 = lower_bound_u64(ix.border_rows, ix.n_border, i);
    return __ldg(ix.count + 5) + (i - rank0 - (lf_sum - counts));
}

// K32: an expansion fetches the record of each border once (one record when both share it) and derives the child
// of every searchable symbol from them, the derived symbol (sigma 6 with `N` searchable) included
struct HammingK32Source {
    const DevIndex &ix;
    uint32_t ns;
    uint64_t n;
    struct Node {
        uint64_t s[5], e[5];
    };
    __device__ __forceinline__ void expand(uint64_t s, uint64_t e, Node &nd) const {
        const K32::Rec rs = K32::load(ix, s, 0);
        const K32::Rec re = (s >> 6) == (e >> 6) ? rs : K32::load(ix, e, 0);
        uint64_t sum_s = 0, sum_e = 0;
#pragma unroll
        for (uint32_t c = 1; c <= 4; ++c) {
            if (c > ns) break;
            nd.s[c - 1] = sbc_load(ix, s, c) + K32::local_rank(rs, c, s);
            nd.e[c - 1] = sbc_load(ix, e, c) + K32::local_rank(re, c, e);
            sum_s += nd.s[c - 1];
            sum_e += nd.e[c - 1];
        }
        if (ns > 4) {
            nd.s[4] = k32_lf_derived_from_sum(ix, s, sum_s);
            nd.e[4] = k32_lf_derived_from_sum(ix, e, sum_e);
        }
    }
    __device__ __forceinline__ void child(const Node &nd, uint32_t c, uint64_t &s, uint64_t &e) const {
        s = nd.s[c - 1];
        e = nd.e[c - 1];
    }
    __device__ __forceinline__ void step(uint32_t c, uint64_t &s, uint64_t &e) const { lf_pair<K32>(ix, c, s, e); }
};

// KG<B> (up to 255 searchable symbols): a node keeps its interval, each child costs one LF pair when it is tried
template <class L>
struct HammingLazySource {
    const DevIndex &ix;
    uint32_t ns;
    uint64_t n;
    struct Node {
        uint64_t s, e;
    };
    __device__ __forceinline__ void expand(uint64_t s, uint64_t e, Node &nd) const {
        nd.s = s;
        nd.e = e;
    }
    __device__ __forceinline__ void child(const Node &nd, uint32_t c, uint64_t &s, uint64_t &e) const {
        s = nd.s;
        e = nd.e;
        lf_pair<L>(ix, c, s, e);
    }
    __device__ __forceinline__ void step(uint32_t c, uint64_t &s, uint64_t &e) const { lf_pair<L>(ix, c, s, e); }
};

template <class L>
struct HammingSourceOf {
    using type = HammingLazySource<L>;
};
template <>
struct HammingSourceOf<K32> {
    using type = HammingK32Source;
};

// dense symbol of query position j (IO bytes through the shared translation table)
struct HammingQuery {
    const uint8_t *tab, *p;
    __device__ __forceinline__ uint32_t operator()(uint32_t j) const { return tab[__ldg(p + j)]; }
};

// PASS 1: checks every query in full (every byte must be a searchable symbol), then writes occ[q * (k + 1) + d]
// (occurrences with exactly d mismatches) and, with n_iv, the number of intervals of query q; counts the node
// expansions into *stat_expansions.  PASS 2: runs the same search again and writes the intervals of query q from
// iv_off[q] on as sort keys and values (HammingWriter).  One thread per query; the frame stack (hamming.h) lives in
// local memory.
template <class L, int PASS>
__global__ void __launch_bounds__(256)
k_hamming(const __grid_constant__ DevIndex ix, const DevQueries qs, uint32_t k, uint64_t q_index_base, uint64_t *err,
          uint64_t *__restrict__ occ, uint64_t *__restrict__ n_iv, const uint64_t *__restrict__ iv_off,
          uint64_t *__restrict__ keys, uint64_t *__restrict__ vals, unsigned long long *stat_expansions) {
    __shared__ uint8_t tab[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = ix.io_to_dense[i];
    __syncthreads();
    using S = typename HammingSourceOf<L>::type;
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t expansions = 0;
    if (q < qs.nq) {
        uint64_t begin, len;
        query_extent(qs, q, begin, len);
        const S rs{ix, ix.ns, ix.n};
        const HammingQuery sym{tab, qs.bytes + begin};
        HammingFrame<typename S::Node> stack[kHammingMaxQueryLen];
        if constexpr (PASS == 1) {
            // (the host refuses broken offsets and long queries before the search; this keeps such a query from
            // being read out of bounds all the same)
            const bool broken = begin > qs.limit || len > qs.limit - begin;
            bool bad = broken || len > kHammingMaxQueryLen;
            for (uint32_t j = 0; !bad && j < len; ++j) {
                const uint32_t c = sym(j);
                bad = c == 0 || c > ix.ns;
            }
            HammingCounter cnt;
            if (bad) report_error(err, (broken ? kBadOffsetFlag : 0ull) | (q_index_base + q));
            else expansions = hamming_search(rs, sym, (uint32_t)len, k, stack, cnt);
            for (uint32_t d = 0; d <= k; ++d) occ[q * (k + 1) + d] = cnt.occ[d];
            if (n_iv) n_iv[q] = cnt.intervals;
        } else {
            HammingWriter w{keys, vals, iv_off[q]};
            hamming_search(rs, sym, (uint32_t)len, k, stack, w);
        }
    }
    if (PASS == 1 && stat_expansions) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) expansions += __shfl_down_sync(0xffffffffu, expansions, o);
        if ((threadIdx.x & 31) == 0 && expansions) atomicAdd(stat_expansions, (unsigned long long)expansions);
    }
}

// the pairs of pass 2, sorted by start per query -> records (iv) or interval ends (the starts are the keys)
__global__ void k_hamming_decode(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals, uint64_t n,
                                 HammingInterval *__restrict__ iv, uint64_t *__restrict__ ends) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const HammingInterval h = hamming_decode(keys[i], vals[i]);
    if (iv) iv[i] = h;
    else ends[i] = h.end;
}

// out[i] = src[idx[i]], i < n (hit offsets of a query = those of its first interval)
__global__ void k_gather_u64(const uint64_t *__restrict__ idx, const uint64_t *__restrict__ src, uint64_t n,
                             uint64_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[idx[i]];
}

// ---- CSR plumbing for locate --------------------------------------------------------------------------
constexpr uint32_t kExpandInline = 32;
constexpr uint64_t kResolvedBit = 1ull << 63;  // rows[] entry is a text position, not an SA row

// counts[q] = width of interval q; *big_count = number of intervals wider than kExpandInline
__global__ void k_interval_counts(const uint64_t *__restrict__ starts, const uint64_t *__restrict__ ends,
                                  uint64_t n, uint64_t *__restrict__ counts,
                                  unsigned long long *big_count) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const uint64_t c = ends[q] == kDirectHit ? 1 : ends[q] - starts[q];
    counts[q] = c;
    if (c > kExpandInline) atomicAdd(big_count, 1ull);
}

// rows[hit_offsets[q] + j] = starts[q] + j; intervals wider than kExpandInline go to a worklist
__global__ void k_expand_rows(const uint64_t *__restrict__ starts, const uint64_t *__restrict__ ends,
                              const uint64_t *__restrict__ hit_offsets, uint64_t n,
                              uint64_t *__restrict__ rows, uint64_t *__restrict__ big_list,
                              unsigned long long *big_cursor) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const uint64_t s = starts[q], off = hit_offsets[q];
    if (ends[q] == kDirectHit) {  // already a text position (verified in k_search): tag it for the walk
        rows[off] = s | kResolvedBit;
        return;
    }
    const uint64_t cnt = ends[q] - s;
    if (cnt > kExpandInline) {
        big_list[atomicAdd(big_cursor, 1ull)] = q;
        return;
    }
    for (uint64_t j = 0; j < cnt; ++j) rows[off + j] = s + j;
}

// chunk-local CSR offsets -> global ones (pipelined locate)
__global__ void k_add_base(uint64_t *__restrict__ offsets, uint64_t n, uint64_t base) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n) offsets[q] += base;
}

// one CTA per wide interval, coalesced fill
__global__ void k_expand_big_rows(const uint64_t *__restrict__ starts, const uint64_t *__restrict__ ends,
                                  const uint64_t *__restrict__ hit_offsets,
                                  const uint64_t *__restrict__ big_list, uint64_t *__restrict__ rows) {
    const uint64_t q = big_list[blockIdx.x];
    const uint64_t s = starts[q], cnt = ends[q] - s, off = hit_offsets[q];
    for (uint64_t j = (uint64_t)blockIdx.y * blockDim.x + threadIdx.x; j < cnt;
         j += (uint64_t)gridDim.y * blockDim.x)
        rows[off + j] = s + j;
}

// a hit as gdx_hit (2 x u64) or, for texts shorter than 2^32, as gdx_hit32 (2 x u32: half the D2H bytes)
__device__ __forceinline__ void store_hit(ulonglong2 *hits, uint64_t h, uint64_t text_id, uint64_t position, int compact) {
    if (compact) reinterpret_cast<uint2 *>(hits)[h] = make_uint2((uint32_t)text_id, (uint32_t)position);
    else hits[h] = make_ulonglong2(text_id, position);
}

// ---- K3 + K4: LF-walk to the next sample, then position -> (text id, position in text) ---------------
template <class L>
__global__ void __launch_bounds__(256)
k_locate_walk(const __grid_constant__ DevIndex ix, const uint64_t *__restrict__ rows, uint64_t nh,
              ulonglong2 *__restrict__ hits, unsigned long long *stat_steps, int compact) {
    const uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t steps = 0;
    if (h < nh) {
        const uint64_t row = rows[h];
        const uint64_t pos = (row & kResolvedBit) ? (row & ~kResolvedBit) : resolve_row<L>(ix, row, steps);
        // text_id_search_tree.rs:35-64: lower_bound over the sentinel positions
        uint64_t id = lower_bound_u64(ix.sentinels, ix.ntexts, pos);
        if (id >= ix.ntexts) id = ix.ntexts - 1;
        const uint64_t base = id == 0 ? 0 : __ldg(ix.sentinels + id - 1) + 1;
        store_hit(hits, h, id, pos - base, compact);
    }
    if (stat_steps) {
        uint32_t tot = __reduce_add_sync(0xffffffffu, steps);
        if ((threadIdx.x & 31) == 0 && tot) atomicAdd(stat_steps, (unsigned long long)tot);
    }
}

// The same with warp-level compaction of finished walks (north-star (3)): with row sampling a walk takes a
// geometric number of LF steps (mean rate - 1, long tail), so in the one-thread-per-hit kernel most lanes of a
// warp idle while its slowest walk finishes.  Here a lane that has finished takes the next unresolved hit of
// its CTA's slice at once (one warp-aggregated atomic per refill), so every lane issues a record fetch in every
// iteration; every hit is still written to its own slot, so the order of the results does not change.
constexpr uint32_t kWalkSlice = 2048;  // hits per CTA slice
template <class L>
__global__ void __launch_bounds__(256)
k_locate_walk_compact(const __grid_constant__ DevIndex ix, const uint64_t *__restrict__ rows, uint64_t nh,
                      ulonglong2 *__restrict__ hits, unsigned long long *stat_steps, int compact) {
    __shared__ uint32_t next;  // next unclaimed hit of the slice
    const uint64_t slice0 = (uint64_t)blockIdx.x * kWalkSlice;
    const uint32_t slice_n = (uint32_t)(nh - slice0 < kWalkSlice ? nh - slice0 : kWalkSlice);
    if (threadIdx.x == 0) next = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    uint64_t h = 0, row = 0;
    uint32_t steps = 0, total_steps = 0;
    bool active = false;
    for (;;) {
        // refill idle lanes
        const uint32_t idle = __ballot_sync(0xffffffffu, !active);
        if (idle) {
            uint32_t base = 0;
            if (lane == (uint32_t)(__ffs(idle) - 1)) base = atomicAdd(&next, (uint32_t)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, __ffs(idle) - 1);
            if (!active) {
                const uint32_t k = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
                if (k < slice_n) {
                    h = slice0 + k;
                    row = rows[h];
                    steps = 0;
                    active = true;
                }
            }
            if (__ballot_sync(0xffffffffu, active) == 0) break;  // slice exhausted and every walk finished
        }
        if (active) {
            // one step of resolve_row (sampled_suffix_array.rs:110-138)
            uint64_t pos = 0;
            bool done = false;
            if (row & kResolvedBit) {
                pos = row & ~kResolvedBit;
                done = true;
            } else {
                const bool sampled = ix.sampling_shift != 0xffffffffu ? (row & ((1ull << ix.sampling_shift) - 1)) == 0
                                                                      : (row % ix.sampling_rate) == 0;
                if (sampled) {
                    const uint64_t k = ix.sampling_shift != 0xffffffffu ? row >> ix.sampling_shift : row / ix.sampling_rate;
                    pos = (ix.wide ? __ldg(reinterpret_cast<const uint64_t *>(ix.samples) + k)
                                   : (uint64_t)__ldg(reinterpret_cast<const uint32_t *>(ix.samples) + k)) + steps;
                    done = true;
                } else {
                    typename L::Planes pl = L::load_planes_once(ix, row);
                    const uint32_t c = L::symbol_at(pl, row);
                    if (c == 0) {  // :121-126 text_border_lookup[&i]
                        const uint64_t k = lower_bound_u64(ix.border_rows, ix.n_border, row);
                        pos = __ldg(ix.border_pos + k) + steps;
                        done = true;
                    } else {
                        if (c > ix.noff) {
                            row = L::lf_derived(ix, row);
                        } else {
                            typename L::Rec r = L::with_offset(ix, pl, row, c);
                            row = sbc_load(ix, row, c) + L::local_rank(r, c, row);
                        }
                        ++steps;
                        ++total_steps;
                    }
                }
            }
            if (done) {
                uint64_t id = lower_bound_u64(ix.sentinels, ix.ntexts, pos);  // text_id_search_tree.rs:35-64
                if (id >= ix.ntexts) id = ix.ntexts - 1;
                const uint64_t base = id == 0 ? 0 : __ldg(ix.sentinels + id - 1) + 1;
                store_hit(hits, h, id, pos - base, compact);
                active = false;
            }
        }
    }
    if (stat_steps) {
        const uint32_t tot = __reduce_add_sync(0xffffffffu, total_steps);
        if (lane == 0 && tot) atomicAdd(stat_steps, (unsigned long long)tot);
    }
}

// ---- construction of the derived structures on the device --------------------------------------------
// One CTA per superblock (65536 positions); thread t packs block t.  sb_tot[sb*noff + c-1] receives
// the number of c in the superblock; k_sb_scan turns that into sbc (exclusive prefix + count[c]).
__global__ void __launch_bounds__(1024)
k_pack_k32(const uint8_t *__restrict__ bwt, uint64_t n, uint32_t noff, uint8_t *__restrict__ records,
           uint64_t n_records, uint64_t *__restrict__ sb_tot) {
    using Scan = cub::BlockScan<uint32_t, 1024>;
    __shared__ typename Scan::TempStorage tmp;
    const uint64_t blk = (uint64_t)blockIdx.x * 1024 + threadIdx.x;
    const uint64_t p0 = blk << 6;
    uint64_t w[4] = {0, 0, 0, 0};
    if (p0 < n) {
        const uint32_t nsym = n - p0 < 64 ? (uint32_t)(n - p0) : 64u;
        for (uint32_t j = 0; j < nsym; ++j) {
            const uint32_t s = bwt[p0 + j];
            w[0] |= (uint64_t)(s & 1u) << j;
            w[1] |= (uint64_t)((s >> 1) & 1u) << j;
            w[2] |= (uint64_t)((s >> 2) & 1u) << j;
        }
    }
    for (uint32_t c = 1; c <= noff; ++c) {
        // positions >= n hold all-zero planes = symbol 0, so they never match c >= 1
        uint32_t cnt = (uint32_t)popc64(match_planes<3>(w, c)), excl, total;
        Scan(tmp).ExclusiveSum(cnt, excl, total);
        __syncthreads();
        w[3] |= (uint64_t)(excl & 0xffffu) << (16u * (c - 1u));
        if (threadIdx.x == 0) sb_tot[(uint64_t)blockIdx.x * noff + (c - 1)] = total;
    }
    if (blk < n_records) {
        uint4 *dst = reinterpret_cast<uint4 *>(records + (blk << 5));
        dst[0] = make_uint4((uint32_t)w[0], (uint32_t)(w[0] >> 32), (uint32_t)w[1], (uint32_t)(w[1] >> 32));
        dst[1] = make_uint4((uint32_t)w[2], (uint32_t)(w[2] >> 32), (uint32_t)w[3], (uint32_t)(w[3] >> 32));
    }
}

template <int B>
__global__ void __launch_bounds__(512)
k_pack_kg(const uint8_t *__restrict__ bwt, uint64_t n, uint32_t sigma, uint32_t stride,
          uint8_t *__restrict__ records, uint64_t n_records, uint64_t *__restrict__ sb_tot) {
    using Scan = cub::BlockScan<uint32_t, 512>;
    __shared__ typename Scan::TempStorage tmp;
    const uint64_t blk = (uint64_t)blockIdx.x * 512 + threadIdx.x;
    const uint64_t p0 = blk << 7;
    uint64_t lo[B], hi[B];
#pragma unroll
    for (int p = 0; p < B; ++p) lo[p] = hi[p] = 0;
    if (p0 < n) {
        const uint32_t nsym = n - p0 < 128 ? (uint32_t)(n - p0) : 128u;
        for (uint32_t j = 0; j < nsym; ++j) {
            const uint32_t s = bwt[p0 + j];
#pragma unroll
            for (int p = 0; p < B; ++p) {
                const uint64_t bit = (uint64_t)((s >> p) & 1u) << (j & 63u);
                if (j < 64) lo[p] |= bit; else hi[p] |= bit;
            }
        }
    }
    uint8_t *rec = records + blk * stride;
    const uint32_t noff = sigma - 1;
    for (uint32_t c = 1; c <= noff; ++c) {
        uint32_t cnt = (uint32_t)(popc64(match_planes<B>(lo, c)) + popc64(match_planes<B>(hi, c)));
        uint32_t excl, total;
        Scan(tmp).ExclusiveSum(cnt, excl, total);
        __syncthreads();
        if (blk < n_records) reinterpret_cast<uint16_t *>(rec + 16 * B)[c - 1] = (uint16_t)excl;
        if (threadIdx.x == 0) sb_tot[(uint64_t)blockIdx.x * noff + (c - 1)] = total;
    }
    if (blk < n_records) {
#pragma unroll
        for (int p = 0; p < B; ++p)
            reinterpret_cast<ulonglong2 *>(rec)[p] = make_ulonglong2(lo[p], hi[p]);
    }
}

// in place: sbc[sb][c-1] = count[c] + sum_{sb' < sb} tot[sb'][c-1]   (condensed.rs:104-116 + lib.rs:273-275)
__global__ void k_sb_scan(uint64_t *__restrict__ sbc, uint64_t n_superblocks, uint32_t noff,
                          const uint64_t *__restrict__ count) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;  // symbol c+1
    if (c >= noff) return;
    uint64_t acc = count[c + 1];
    for (uint64_t sb = 0; sb < n_superblocks; ++sb) {
        const uint64_t t = sbc[sb * noff + c];
        sbc[sb * noff + c] = acc;
        acc += t;
    }
}

// lookup_table.rs:225-258: entry i of level d = extend(entry i / ns of level d-1, symbol i % ns + 1)
template <class L>
__global__ void __launch_bounds__(256)
k_lut_fill(const __grid_constant__ DevIndex ix, void *__restrict__ lookup, uint32_t d) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ix.lut_pow[d]) return;
    uint64_t s, e;
    lut_load(ix, ix.lut_level_off[d - 1] + i / ix.ns, s, e);
    const uint32_t c = (uint32_t)(i % ix.ns) + 1;
    if (s != e) lf_pair<L>(ix, c, s, e);  // cursor.rs:40-51
    const uint64_t entry = ix.lut_level_off[d] + i;
    if (ix.wide)
        reinterpret_cast<ulonglong2 *>(lookup)[entry] = make_ulonglong2(s, e);
    else
        reinterpret_cast<uint2 *>(lookup)[entry] = make_uint2((uint32_t)s, (uint32_t)e);
}

// one level of the seed table from the previous one, each in its own buffer (same rule as k_lut_fill)
template <class L>
__global__ void __launch_bounds__(256)
k_lut_extend(const __grid_constant__ DevIndex ix, const void *__restrict__ prev, void *__restrict__ out, uint64_t entries) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= entries) return;
    uint64_t s, e;
    if (ix.wide) {
        const ulonglong2 v = reinterpret_cast<const ulonglong2 *>(prev)[i / ix.ns];
        s = v.x;
        e = v.y;
    } else {
        const uint2 v = reinterpret_cast<const uint2 *>(prev)[i / ix.ns];
        s = v.x;
        e = v.y;
    }
    const uint32_t c = (uint32_t)(i % ix.ns) + 1;
    if (s != e) lf_pair<L>(ix, c, s, e);  // cursor.rs:40-51
    if (ix.wide)
        reinterpret_cast<ulonglong2 *>(out)[i] = make_ulonglong2(s, e);
    else
        reinterpret_cast<uint2 *>(out)[i] = make_uint2((uint32_t)s, (uint32_t)e);
}

// symbol_at over the reference's own block arrays, any of its four rank variants (lib.rs:104-113):
// condensed (condensed.rs:343-362): [group][plane] Blocks of `words` u64, bit j of the group = position j;
// flat (flat.rs:248-267): [group][symbol] one-hot Blocks, position j at bit j + 16 (block.rs:3), `used` = NUM_BITS - 16
__global__ void k_ref_blocks_to_bwt(const uint64_t *__restrict__ blocks, uint32_t flat, uint32_t words, uint32_t units,
                                    uint64_t n, uint8_t *__restrict__ bwt) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t used = words * 64 - (flat ? 16 : 0);
    const uint64_t g = i / used;
    const uint32_t bit = (uint32_t)(i % used) + (flat ? 16 : 0);
    const uint64_t *grp = blocks + g * units * words + bit / 64;
    uint32_t s = 0;
    if (flat) {
        for (uint32_t c = 0; c < units; ++c)
            if ((grp[(uint64_t)c * words] >> (bit & 63)) & 1u) s = c;
    } else {
        for (uint32_t p = 0; p < units; ++p) s |= (uint32_t)((grp[(uint64_t)p * words] >> (bit & 63)) & 1u) << p;
    }
    bwt[i] = (uint8_t)s;
}

// symbol_at over the device records: the dense BWT back (export utility)
template <class L>
__global__ void __launch_bounds__(256)
k_records_to_bwt(const __grid_constant__ DevIndex ix, uint64_t begin, uint64_t end, uint8_t *__restrict__ out) {
    const uint64_t i = begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= end) return;
    typename L::Planes pl = L::load_planes(ix, i);
    out[i - begin] = (uint8_t)L::symbol_at(pl, i);
}

// dense text -> text section: two symbols per byte (low nibble = even position) or a plain copy
__global__ void k_pack_text(const uint8_t *__restrict__ text, uint64_t n, uint32_t bits, uint8_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (bits == 4) {
        if (2 * i >= n) return;
        const uint32_t lo = text[2 * i], hi = 2 * i + 1 < n ? text[2 * i + 1] : 0;
        out[i] = (uint8_t)(lo | (hi << 4));
    } else if (i < n) {
        out[i] = text[i];
    }
}

__global__ void k_widen_u32(const uint32_t *__restrict__ in, uint64_t n, uint64_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}
__global__ void k_narrow_u64(const uint64_t *__restrict__ in, uint64_t n, uint32_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint32_t)in[i];
}

// ---- dense suffix array accelerator: SA[row] for every row from the sampled one (one walk per row) -----
template <class L>
__global__ void __launch_bounds__(256)
k_densify(const __grid_constant__ DevIndex ix, void *__restrict__ out, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t steps = 0;
    const uint64_t v = resolve_row<L>(ix, i, steps);
    if (ix.wide) reinterpret_cast<uint64_t *>(out)[i] = v;
    else reinterpret_cast<uint32_t *>(out)[i] = (uint32_t)v;
}

// ---- row context table: SA[row] + the 45 text symbols in front of it (layout: see ctx_matches) ------------
template <class L>
__global__ void __launch_bounds__(256)
k_build_row_context(const __grid_constant__ DevIndex ix, uint4 *__restrict__ out, uint64_t n) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    uint32_t steps = 0;
    const uint64_t at = resolve_row<L>(ix, row, steps);
    const CtxEntry en = ctx_make_entry(at, ix.ns, [&](uint64_t p) { return text_symbol(ix, p); });
    out[row] = make_uint4(en.x, en.y, en.z, en.w);
}

// ---- random-gather ceiling (SURVEY 8d) ----------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t x) {  // splitmix64 finalizer
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

// every thread issues `rounds` x 2 loads of REC bytes at pseudo-random record indices
// (the table holds record_mask + 1 = a power of two records).
// chained = 0: addresses depend only on a counter (pure bandwidth / MLP ceiling);
// chained = 1: the next pair of addresses depends on the loaded data, like an LF step.
template <int REC>
__global__ void __launch_bounds__(256)
k_gather(const uint8_t *__restrict__ table, uint64_t record_mask, uint32_t rounds, int chained,
         uint64_t *__restrict__ sink) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t a = mix64(tid * 2 + 1), b = mix64(tid * 2 + 2), acc = 0;
    for (uint32_t r = 0; r < rounds; ++r) {
        const uint8_t *pa = table + (a & record_mask) * REC, *pb = table + (b & record_mask) * REC;
        uint64_t wa[4], wb[4];
        if (REC == 32) {
            ldg256_na(pa, wa);
            ldg256_na(pb, wb);
        } else {
            uint64_t t0[4], t1[4];
            ldg256_na(pa, wa);
            ldg256_na(pa + 32, t0);
            ldg256_na(pb, wb);
            ldg256_na(pb + 32, t1);
            wa[0] ^= t0[0] ^ t0[3];
            wb[0] ^= t1[0] ^ t1[3];
            if (REC == 128) {
                ldg256_na(pa + 64, t0);
                ldg256_na(pa + 96, t1);
                wa[1] ^= t0[1] ^ t1[2];
                ldg256_na(pb + 64, t0);
                ldg256_na(pb + 96, t1);
                wb[1] ^= t0[1] ^ t1[2];
            }
        }
        const uint64_t xa = wa[0] ^ wa[1] ^ wa[2] ^ wa[3], xb = wb[0] ^ wb[1] ^ wb[2] ^ wb[3];
        acc += xa + xb;
        if (chained) {
            a = mix64(a ^ xa);
            b = mix64(b ^ xb);
        } else {
            a = mix64(a);
            b = mix64(b);
        }
    }
    if (acc == 0x1234567812345678ull) sink[0] = acc;  // keep the loads alive
}

}  // namespace gdx
#endif
