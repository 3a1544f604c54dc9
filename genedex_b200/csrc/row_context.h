// row_context.h -- bit layout of the row context table and of 2-bit coded queries (accelerator,
// gdx_index_set_row_context_table).  Like rank_core.h everything here is __host__ __device__, so that
// tests/host_emul can run the exact arithmetic of the kernels on the CPU against a plain model.
//
// One 16-byte entry per suffix array row:
//   x                    SA[row]
//   y | z << 32 | w << 64  96 bits; bits [2i, 2i + 2), i = 0..44: 2-bit code (dense - 1) of text[SA[row] - 45 + i];
//                        top 6 bits of w: vl = number of symbols directly in front of SA[row] that are searchable
//                        symbols of the same text (0..45); codes outside that run are 0 and must not be compared
// A one-row interval with at most vl query symbols left is verified from this one entry -- one random DRAM line
// instead of the suffix array entry plus the text window behind it.  Alphabets with at most 4 searchable symbols,
// texts shorter than 2^32 symbols.
#ifndef GDX_ROW_CONTEXT_H
#define GDX_ROW_CONTEXT_H

#include <stdint.h>

#include "rank_core.h"

namespace gdx {

constexpr uint32_t kCtxSymbols = 45;

struct CtxEntry {
    uint32_t x, y, z, w;
};

// 2-bit form of (the last 64 symbols of) a query: symbol j at bits [2j, 2j + 2) of the 128-bit value hi:lo
struct PackedTail {
    uint64_t lo, hi;
};

GDX_HD uint32_t ctx_valid_len(const CtxEntry &en) { return en.w >> 26; }

// text_symbol(p) = dense symbol at text position p; at = SA[row]; ns = number of searchable symbols (<= 4)
template <class TextSymbol>
GDX_HD CtxEntry ctx_make_entry(uint64_t at, uint32_t ns, TextSymbol text_symbol) {
    uint32_t w0 = 0, w1 = 0, w2 = 0, vl = 0;
    for (uint32_t k = 1; k <= kCtxSymbols && k <= at; ++k) {  // text position at - k <-> code index 45 - k
        const uint32_t d = text_symbol(at - k);
        if (d == 0 || d > ns) break;
        const uint32_t i = kCtxSymbols - k, bits = (d - 1) << ((i & 15) * 2);
        if (i < 16) w0 |= bits;
        else if (i < 32) w1 |= bits;
        else w2 |= bits;
        vl = k;
    }
    return CtxEntry{(uint32_t)at, w0, w1, w2 | (vl << 26)};
}

// query[0..pos) (codes at bits [2j, 2j + 2) of qh:ql) against the last pos (1..vl) symbols of the entry
GDX_HD bool ctx_matches(const CtxEntry &en, uint32_t pos, uint64_t ql, uint64_t qh) {
    const uint64_t lo = (uint64_t)en.y | ((uint64_t)en.z << 32), hi = en.w & 0x3ffffffu;
    const uint32_t sh = 2 * (kCtxSymbols - pos);  // the symbol that meets query[0] moves to bit 0
    uint64_t rl, rh;
    if (sh == 0) {
        rl = lo;
        rh = hi;
    } else if (sh < 64) {
        rl = (lo >> sh) | (hi << (64 - sh));
        rh = hi >> sh;
    } else {
        rl = hi >> (sh - 64);
        rh = 0;
    }
    const uint32_t nb = 2 * pos;
    const uint64_t ml = nb >= 64 ? ~0ull : (1ull << nb) - 1, mh = nb > 64 ? (1ull << (nb - 64)) - 1 : 0ull;
    return (((rl ^ ql) & ml) | ((rh ^ qh) & mh)) == 0;
}

// bytes mis .. mis + 3 of the little-endian byte string w0 w1
GDX_HD uint32_t bytes_at(uint32_t w0, uint32_t w1, uint32_t mis) {
#ifdef __CUDA_ARCH__
    return __byte_perm(w0, w1, 0x3210u + 0x1111u * mis);
#else
    return (uint32_t)((((uint64_t)w1 << 32) | w0) >> (8 * mis));
#endif
}

// IO-byte queries of an alphabet with at most 4 searchable symbols are turned into the 2-bit form of the packed
// kernel right after staging, four bytes at a time: tab2[b] = dense - 1 for a searchable byte, 0x100 for every other
// one.  slot = the staged words (the kernel's shared-memory slot), the query bytes start at byte `mis` (0..3) of it;
// tail <= 64 symbols; slot[(mis + tail + 3) / 4] and the words behind it may hold anything (never dereferenced past
// word 16).  Returns false (t unspecified) if a staged byte is not a searchable symbol: such a query keeps the
// byte-wise path with its lazy error behaviour.  ~5 instructions per symbol once, instead of a table walk per
// symbol per use.
GDX_HD bool codes_from_staged(const uint16_t *tab2, const uint32_t *slot, uint32_t mis, uint32_t tail, PackedTail &t) {
    uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0, flags = 0;
    uint32_t w0 = slot[0];
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (uint32_t k = 0; k < 16; ++k) {
        if (4 * k < tail) {
            const uint32_t w1 = slot[k + 1];
            const uint32_t w = bytes_at(w0, w1, mis);
            w0 = w1;
            // codes of the four symbols in bits 0..7, their "not searchable" flags in bits 8, 10, 12, 14
            uint32_t x = (uint32_t)tab2[w & 0xffu] + 4u * tab2[(w >> 8) & 0xffu] + 16u * tab2[(w >> 16) & 0xffu] +
                         64u * tab2[w >> 24];
            const uint32_t cnt = tail - 4 * k;  // symbols of this word that belong to the query
            if (cnt < 4) x &= 0x0101u * ((1u << (2 * cnt)) - 1u);
            flags |= x;
            const uint32_t bits = (x & 0xffu) << (8 * (k & 3));
            if (k < 4) c0 |= bits;
            else if (k < 8) c1 |= bits;
            else if (k < 12) c2 |= bits;
            else c3 |= bits;
        }
    }
    t.lo = (uint64_t)c0 | ((uint64_t)c1 << 32);
    t.hi = (uint64_t)c2 | ((uint64_t)c3 << 32);
    return (flags >> 8) == 0;
}

// true if one of the first nsym (<= 64) codes of t is >= ns, i.e. not a searchable symbol (dense = code + 1 > ns).
// A caller's pre-packed batch can hold such codes when the alphabet has fewer than 4 searchable symbols; every code
// is searchable when ns >= 4.  Codes past nsym are ignored.
GDX_HD bool packed_codes_unsearchable(const PackedTail &t, uint32_t nsym, uint32_t ns) {
    if (ns >= 4 || nsym == 0) return false;
    const uint64_t ml = nsym >= 32 ? ~0ull : (1ull << (2 * nsym)) - 1ull;
    const uint64_t mh = nsym >= 64 ? ~0ull : (nsym > 32 ? (1ull << (2 * (nsym - 32))) - 1ull : 0ull);
    // bit 2j of a word is set if code j of it is out of range: ns 1 -> code != 0, 2 -> high bit, 3 -> both bits
    auto out = [ns](uint64_t x) {
        const uint64_t lo = x & 0x5555555555555555ull, hi = (x >> 1) & 0x5555555555555555ull;
        return ns == 1 ? (lo | hi) : (ns == 2 ? hi : (lo & hi));
    };
    return ((out(t.lo) & ml) | (out(t.hi) & mh)) != 0;
}

// tab2 of codes_from_staged from the alphabet's translation table
GDX_HD uint16_t ctx_tab2_entry(uint32_t dense, uint32_t ns) { return (uint16_t)((dense >= 1 && dense <= ns) ? dense - 1 : 0x100u); }

}  // namespace gdx
#endif
