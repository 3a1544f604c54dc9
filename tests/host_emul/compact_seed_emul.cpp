// Host build of the compact seed level (genedex_b200/csrc/compact_seed.h) and its policy (accel_policy.h) for
// tests/test_compact_seed_host.py.  cs_build lays out the table the way the device builder does (groups, then the
// exception records in d-mer order), from a suffix array and the dense text, with the header's row key.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../genedex_b200/csrc/accel_policy.h"
#include "../../genedex_b200/csrc/compact_seed.h"

extern "C" uint64_t emul_cs_index_from_codes(uint64_t v, uint32_t d) { return gdx::cs_index_from_codes(v, d); }

extern "C" void emul_cs_decode(const uint64_t *w, uint32_t j, const uint32_t *pool, uint64_t *out) {
    gdx::cs_decode(w, j, pool, out[0], out[1]);
}

// groups: cs_groups(ns^d) * 64 bytes; pool: room for 4 n + 4 words.  Returns the pool words used, or -1 if the keys
// decrease along the suffix array or a gap row comes before a row with the prefix of the same d-mer.
extern "C" int64_t emul_cs_build(const uint8_t *text, uint64_t n, const uint32_t *sa, uint32_t d, uint32_t ns,
                                 uint8_t *groups, uint32_t *pool) {
    uint64_t kmers = 1;
    for (uint32_t i = 0; i < d; ++i) kmers *= ns;
    const uint64_t G = gdx::cs_groups(kmers);
    std::vector<uint64_t> code(n);
    for (uint64_t r = 0; r < n; ++r) {
        const uint64_t at = sa[r];
        bool gap = false;
        const uint64_t k1 = gdx::cs_row_key([&](uint32_t j) { return at + j < n ? (uint32_t)text[at + j] : 0u; }, d, ns, gap);
        code[r] = 2 * k1 + (gap ? 1 : 0);
        if (r && code[r] < code[r - 1]) return -1;
    }
    std::memset(groups, 0, G * gdx::kCsGroupBytes);
    uint64_t r = 0;
    for (uint64_t g = 0; g < G; ++g) {
        while (r < n && (code[r] >> 1) <= gdx::kCsSlots * g) ++r;
        uint32_t hdr[2] = {(uint32_t)r, gdx::kCsNoRecord};
        std::memcpy(groups + g * gdx::kCsGroupBytes, hdr, 8);
    }
    int64_t used = 0;
    uint64_t cur_group = ~0ull;
    uint32_t cur_off = 0;
    for (uint64_t a = 0; a < n;) {
        const uint64_t k1 = code[a] >> 1;
        uint64_t b = a, width = 0, gap = 0;
        while (b < n && (code[b] >> 1) == k1) {
            if (code[b] & 1) ++gap;
            else if (gap) return -1;
            else ++width;
            ++b;
        }
        if (k1 > 0) {
            const uint64_t k = k1 - 1, g = k / gdx::kCsSlots;
            const uint32_t j = (uint32_t)(k % gdx::kCsSlots);
            uint8_t *grp = groups + g * gdx::kCsGroupBytes;
            uint32_t w;
            std::memcpy(&w, grp + 8 + 4 * (j / 16), 4);
            w |= (uint32_t)(width < 3 ? width : 3) << (2 * (j % 16));
            std::memcpy(grp + 8 + 4 * (j / 16), &w, 4);
            if (width >= 3 || gap > 0) {
                if (g != cur_group) {  // the group's record starts here
                    cur_group = g;
                    cur_off = (uint32_t)used;
                    std::memcpy(grp + 4, &cur_off, 4);
                    pool[used++] = 0;
                }
                pool[cur_off]++;
                pool[used++] = j;
                pool[used++] = (uint32_t)width;
                pool[used++] = (uint32_t)gap;
            }
        }
        a = b;
    }
    return used;
}

// {possible, max_depth, fits(d, record_bytes)} of the policy into out
extern "C" void emul_cs_policy(uint64_t n, uint64_t budget, uint32_t ns, int wide, int text, uint32_t seed_depth,
                               uint32_t d, uint64_t record_bytes, uint64_t used, uint64_t free, uint64_t *out) {
    const gdx::AccelPolicy p{n, budget, ns, 0, wide != 0, text != 0, false, false, false};
    out[0] = p.compact_seed_possible(seed_depth);
    out[1] = p.compact_seed_max_depth(seed_depth);
    out[2] = p.compact_seed_fits(d, record_bytes, used, free);
}
