// device_index.h -- the device image of an index: one contiguous allocation + a POD header.
//
// HBM layout (all sections 256 B aligned inside one cudaMalloc'ed arena, so that a replica is one
// ncclBroadcast / one peer copy):
//   records      rank records (rank_core.h), ceil((n+1)/P) * stride bytes   <- random 32/64/128 B
//   sbc          u64 [num_superblocks][noff]: count[c] + #c before the superblock (L2 resident)
//   samples      SA[0], SA[s], SA[2s], ... as u32 (n < 2^32) or u64
//   lookup       all lookup-table levels 0..D back to back, (start,end) pairs of u32 or u64
//   border_rows  sorted SA rows i with BWT[i] == sentinel        (text_border_lookup keys)
//   border_pos   SA[i] for those rows                            (text_border_lookup values)
//   sentinels    sorted sentinel positions of the concatenated text (text id mapping)
//   count        u64 [sigma + 1]  (src/lib.rs:95), only the rare derived-rank path reads it
//   text         (optional) the concatenated dense text, 4 bits per symbol (sigma <= 16) or 8: lets
//                count/locate finish a query whose interval has narrowed to one row by one text
//                comparison instead of one random rank record per remaining symbol
//   isa          (optional, with text) ISA[0], ISA[s], ISA[2s], ...: the SA row of every s-th text position;
//                lets cursors_for_many_queries turn a verified text position back into its interval
#ifndef GDX_DEVICE_INDEX_H
#define GDX_DEVICE_INDEX_H

#include <stdint.h>

#include "rank_core.h"

namespace gdx {

constexpr uint64_t kImageMagic = 0x3130305842584447ull;  // "GDXBX001"
constexpr uint32_t kMaxLookupDepth = 24;
constexpr uint32_t kAccelNoDenseSA = 1, kAccelNoSeedTable = 2, kAccelNoRowContext = 4;

struct ImageHeader {
    uint64_t magic;
    uint32_t version;
    uint32_t wide;  // samples / lookup entries are 64 bit
    uint64_t n;     // text length incl. sentinels
    uint64_t ntexts;
    uint64_t n_border;
    uint64_t n_samples;
    uint64_t n_records;
    uint64_t n_superblocks;
    uint32_t sigma, ns, storage, sampling_rate, lookup_depth;
    uint32_t accel_flags;  // kAccelNoDenseSA | kAccelNoSeedTable | kAccelNoRowContext: accelerator policy, travels with the image
    RankLayout layout;
    uint64_t off_records, off_sbc, off_samples, off_lookup, off_border_rows, off_border_pos,
        off_sentinels, off_count, off_text;
    uint32_t text_bits;  // 0 = no text section, 4 or 8
    uint32_t has_isa;    // sampled inverse suffix array present
    uint64_t off_isa;
    uint64_t accel_budget;  // bytes the accelerators of a replica may take together, 0 = automatic
    uint64_t image_bytes;
    uint64_t lut_level_off[kMaxLookupDepth + 1];  // entry offset of level d
    uint64_t lut_pow[kMaxLookupDepth + 1];        // ns^d
    uint8_t io_to_dense[256];
};

// what the kernels see (passed by value as a __grid_constant__ parameter)
struct DevIndex {
    const uint8_t *records;
    const uint64_t *sbc;
    const void *samples;
    const void *lookup;
    const uint64_t *border_rows;
    const uint64_t *border_pos;
    const uint64_t *sentinels;
    const uint64_t *count;
    const uint8_t *text;
    const void *isa;  // sampled inverse suffix array (same element width as samples) or nullptr
    const void *seed_lookup;  // level seed_depth of a lookup table deeper than the configured one, or nullptr
    const void *row_context;  // 16-byte entries: SA[row] + 45 symbols of text context per row (kernels.cuh: ctx_matches), or nullptr
    const uint8_t *compact_seed;   // groups of the compact seed level (compact_seed.h), or nullptr
    const uint32_t *compact_pool;  // its exception records
    uint64_t n, ntexts, n_border;
    uint32_t sigma, ns, sampling_rate, lookup_depth;
    uint32_t wide, noff, stride, derived_symbol;
    uint32_t sampling_shift;  // log2(sampling_rate) if it is a power of two, else 0xffffffff
    uint32_t text_bits;
    // samples / sampling_rate / sampling_shift describe what resolve_row reads: the image's sampled suffix
    // array, or the dense accelerator (rate 1) once gdx_index_set_dense_suffix_array has built it
    uint32_t verify_min_remaining;  // text verification needs at least this many symbols left (8; 4 with the dense suffix array)
    uint32_t isa_rate;              // sampling rate of the inverse samples (= the configured rate)
    uint32_t seed_depth;
    uint32_t compact_depth;
    uint64_t lut_level_off[kMaxLookupDepth + 1];
    uint64_t lut_pow[kMaxLookupDepth + 1];
    uint8_t io_to_dense[256];
};

inline DevIndex make_dev_index(const ImageHeader &h, const void *image) {
    const uint8_t *base = (const uint8_t *)image;
    DevIndex d;
    d.records = base + h.off_records;
    d.sbc = (const uint64_t *)(base + h.off_sbc);
    d.samples = base + h.off_samples;
    d.lookup = base + h.off_lookup;
    d.border_rows = (const uint64_t *)(base + h.off_border_rows);
    d.border_pos = (const uint64_t *)(base + h.off_border_pos);
    d.sentinels = (const uint64_t *)(base + h.off_sentinels);
    d.count = (const uint64_t *)(base + h.off_count);
    d.text = h.text_bits ? base + h.off_text : nullptr;
    d.text_bits = h.text_bits;
    d.isa = h.has_isa ? base + h.off_isa : nullptr;
    d.n = h.n;
    d.ntexts = h.ntexts;
    d.n_border = h.n_border;
    d.sigma = h.sigma;
    d.ns = h.ns;
    d.sampling_rate = h.sampling_rate;
    d.lookup_depth = h.lookup_depth;
    d.wide = h.wide;
    d.noff = h.layout.noff;
    d.stride = h.layout.stride;
    d.derived_symbol = h.layout.derived_symbol;
    d.sampling_shift = 0xffffffffu;
    d.verify_min_remaining = 8;
    d.isa_rate = h.sampling_rate;
    d.seed_lookup = nullptr;
    d.seed_depth = 0;
    d.row_context = nullptr;
    d.compact_seed = nullptr;
    d.compact_pool = nullptr;
    d.compact_depth = 0;
    if ((h.sampling_rate & (h.sampling_rate - 1)) == 0) {
        uint32_t s = 0;
        while ((1u << s) < h.sampling_rate) ++s;
        d.sampling_shift = s;
    }
    for (uint32_t i = 0; i <= kMaxLookupDepth; ++i) {
        d.lut_level_off[i] = h.lut_level_off[i];
        d.lut_pow[i] = h.lut_pow[i];
    }
    for (int i = 0; i < 256; ++i) d.io_to_dense[i] = h.io_to_dense[i];
    return d;
}

}  // namespace gdx
#endif
