// compact_seed.h -- format of the compact seed level (accelerator, built with the seed table): the suffix array interval
// of every d-mer, d two or more symbols deeper than the seed table, in about 2 bits per d-mer.  Like row_context.h
// everything here is __host__ __device__, so that tests/host_emul runs the exact arithmetic of the kernels on the CPU.
//
// d-mer X = x_0 .. x_{d-1} (x_0 the leftmost of a query's last d symbols) has the index idx = sum (x_j - 1) ns^(d-1-j):
// suffix array order, first symbol most significant.  For d-mer i let S(i) = number of rows whose suffix sorts before
// K_i, width(i) = number of rows with prefix K_i (its interval is [S(i), S(i) + width(i))), gap(i) = S(i+1) - S(i) -
// width(i) with S(last + 1) = n: rows with a sentinel or a non-searchable symbol among their first d symbols
// (cs_row_key says where they sort).
//
// Groups of 224 consecutive d-mers, 64 B each (one DRAM line per lookup):
//   u32 base   S(224 g)
//   u32 exc    word offset of the group's exception record in the pool behind the groups, or kCsNoRecord
//   56 B       224 2-bit fields, slot j at bits [2 (j % 32), 2 (j % 32) + 2) of u64 word 1 + j / 32:
//              f_j = width if width <= 2, else 3
// A group has an exception record when one of its slots has width >= 3 or gap > 0: u32 count, then one
// (slot, width, gap) u32 triple per such slot, slots ascending.  start(j) = base + sum_{i<j} (width_i + gap_i).
#ifndef GDX_COMPACT_SEED_H
#define GDX_COMPACT_SEED_H

#include <stdint.h>

#include "rank_core.h"

namespace gdx {

constexpr uint32_t kCsSlots = 224;       // d-mers per group
constexpr uint32_t kCsGroupBytes = 64;
constexpr uint32_t kCsNoRecord = 0xffffffffu;

GDX_HD uint64_t cs_groups(uint64_t kmers) { return (kmers + kCsSlots - 1) / kCsSlots; }

GDX_HD uint32_t cs_ld(const uint32_t *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// SA-order index of d (1..32) 2-bit codes (dense - 1; ns = 4), code j (x_j) at bits [2j, 2j + 2) of v: the digits of v
// in reverse order
GDX_HD uint64_t cs_index_from_codes(uint64_t v, uint32_t d) {
#ifdef __CUDA_ARCH__
    uint64_t r = __brevll(v);
#else
    uint64_t r = 0;
    for (int b = 0; b < 64; ++b) r |= ((v >> b) & 1ull) << (63 - b);
#endif
    r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);  // bit-reversed pairs back in order
    return r >> (64 - 2 * d);
}

// (start, end) of slot j of a group: w = its 8 little-endian u64 words, pool = the exception records
GDX_HD void cs_decode(const uint64_t w[8], uint32_t j, const uint32_t *pool, uint64_t &s, uint64_t &e) {
    const uint32_t wj = j >> 5, bj = (j & 31u) * 2;
    uint64_t sum = 0, f = 0;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (uint32_t k = 0; k < 7; ++k) {
        const uint64_t x = w[1 + k];
        const uint64_t m = k < wj ? ~0ull : (k == wj ? (1ull << bj) - 1ull : 0ull);
        sum += popc64(x & m) + popc64(x & m & 0xaaaaaaaaaaaaaaaaull);  // sum of the 2-bit fields below slot j
        if (k == wj) f = (x >> bj) & 3u;
    }
    const uint32_t exc = (uint32_t)(w[0] >> 32);
    if (exc != kCsNoRecord) {
        const uint32_t *r = pool + exc;
        const uint32_t cnt = cs_ld(r);
        for (uint32_t i = 0; i < cnt; ++i) {
            const uint32_t slot = cs_ld(r + 1 + 3 * i);
            if (slot > j) break;
            const uint64_t width = cs_ld(r + 2 + 3 * i);
            if (slot == j) {
                f = width;
                break;
            }
            sum += width + cs_ld(r + 3 + 3 * i) - (width < 3 ? width : 3);
        }
    }
    s = (uint32_t)w[0] + sum;
    e = s + f;
}

// Where a suffix sorts among the d-mers.  sym(j) = dense symbol j of the suffix (0 = sentinel, also past the end of the
// text).  Returns key + 1, key = the d-mer the row belongs to (key -1: before d-mer 0), and gap = false when the row
// has that d-mer as its prefix.  With P = the searchable prefix of length j < d in front of the first other symbol x:
//   x the sentinel: the row sorts just before P A^(d-j), a gap row of the d-mer in front of that one;
//   x not searchable: the row sorts after P T^(d-j), a gap row of that d-mer (j = 0: all of them are gaps of the last).
// key + 1 does not decrease from one suffix array row to the next; within a key the rows with the prefix come first.
template <class Sym>
GDX_HD uint64_t cs_row_key(Sym sym, uint32_t d, uint32_t ns, bool &gap) {
    uint64_t idx = 0;
    for (uint32_t j = 0; j < d; ++j) {
        const uint32_t c = sym(j);
        if (c == 0 || c > ns) {
            uint64_t p = 1;
            for (uint32_t k = j; k < d; ++k) p *= ns;
            gap = true;
            return (c == 0 ? idx : idx + 1) * p;
        }
        idx = idx * ns + (c - 1);
    }
    gap = false;
    return idx + 1;
}

}  // namespace gdx
#endif
