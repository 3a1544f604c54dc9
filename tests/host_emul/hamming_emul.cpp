// Host emulation of the Hamming search (genedex_b200/csrc/hamming.h) over the emulated rank records of emul.cpp.
// TEST INFRASTRUCTURE: one shared library with everything of emul.cpp plus emul_hamming, so that the search core k_hamming
// runs can be checked against a naive scan on a machine without a GPU.
#include <algorithm>
#include <utility>

#include "emul.cpp"

// ---- Hamming search over the emulated records ------------------------------------------------------------
#include "../../genedex_b200/csrc/hamming.h"

// emul_lf as the rank source; a node keeps its interval (the lazy form the generic layout uses on the device).
// With `cover` it counts what a test must reach for the device sources to run on inputs where a superblock's
// counts differ from `count`: [0] expansions whose borders lie in different superblocks, [1] children of the derived
// symbol (K32, sigma 6) with a border past superblock 0.
struct EmulHammingSource {
    const void *h;
    uint32_t ns;
    uint64_t n;
    uint64_t *cover;
    struct Node {
        uint64_t s, e;
    };
    void expand(uint64_t s, uint64_t e, Node &nd) const {
        nd.s = s;
        nd.e = e;
        if (cover && (s >> 16) != (e >> 16)) ++cover[0];
    }
    void child(const Node &nd, uint32_t c, uint64_t &s, uint64_t &e) const {
        s = emul_lf(h, c, nd.s);
        e = emul_lf(h, c, nd.e);
        const RankLayout &L = ((const Emul *)h)->L;
        if (cover && L.derived_symbol && c == L.derived_symbol && (nd.e >> 16) > 0) ++cover[1];
    }
    void step(uint32_t c, uint64_t &s, uint64_t &e) const {
        s = emul_lf(h, c, s);
        e = emul_lf(h, c, e);
    }
};

// Both passes of k_hamming for one query of dense symbols (1..ns), m <= kHammingMaxQueryLen, k <= 3, and the sort by
// start that follows them: occ[0..k] = occurrences per number of mismatches; the intervals as (start, end, mismatches)
// triples in iv (up to `cap` of them).  Returns the number of intervals pass 1 counted, or ~0 when pass 2 wrote another
// number; *expansions = node expansions of pass 1.  cover[0..1] are incremented as EmulHammingSource says (pass 1),
// cover[2] once per interval wider than 65 535 rows.
extern "C" uint64_t emul_hamming(const void *h, uint32_t ns, uint64_t n, const uint8_t *query, uint32_t m, uint32_t k,
                                 uint64_t *occ, uint64_t *iv, uint64_t cap, uint64_t *expansions, uint64_t *cover) {
    const EmulHammingSource rs{h, ns, n, cover}, rs2{h, ns, n, nullptr};
    auto sym = [&](uint32_t j) { return (uint32_t)query[j]; };
    std::vector<HammingFrame<EmulHammingSource::Node>> stack(kHammingMaxQueryLen);
    HammingCounter cnt;
    *expansions = hamming_search(rs, sym, m, k, stack.data(), cnt);
    for (uint32_t d = 0; d <= k; ++d) occ[d] = cnt.occ[d];
    std::vector<uint64_t> keys(cnt.intervals + 1), vals(cnt.intervals + 1);
    HammingWriter w{keys.data(), vals.data(), 0};
    hamming_search(rs2, sym, m, k, stack.data(), w);
    if (w.at != cnt.intervals) return ~0ull;
    std::vector<std::pair<uint64_t, uint64_t>> kv;
    for (uint64_t i = 0; i < cnt.intervals; ++i) kv.emplace_back(keys[i], vals[i]);
    std::sort(kv.begin(), kv.end());
    for (uint64_t i = 0; i < cnt.intervals && i < cap; ++i) {
        const HammingInterval x = hamming_decode(kv[i].first, kv[i].second);
        if (x.end - x.start > 65535) ++cover[2];
        iv[3 * i] = x.start;
        iv[3 * i + 1] = x.end;
        iv[3 * i + 2] = x.mismatches;
    }
    return cnt.intervals;
}
