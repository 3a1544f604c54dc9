// Which accelerators an index builds outside its image (include/genedex_b200.h: the dense suffix array, the seed table
// and the row context table) and the text verification threshold that follows from them.  Host only and free of CUDA,
// so that the policy runs on the CPU against a plain model (tests/test_accel_policy_host.py); api.cu observes the free
// device memory and builds the tables.
#pragma once
#include <cstdint>
#include <cstdlib>

namespace gdx {

constexpr uint64_t kFreeUnknown = ~0ull;  // cudaMemGetInfo failed

// entries of level d, 0 if ns^d exceeds 2^36 (grid and memory limits)
inline uint64_t seed_entries(uint32_t ns, uint32_t d) {
    uint64_t e = 1;
    for (uint32_t i = 0; i < d; ++i) {
        e *= ns;
        if (e > (1ull << 36)) return 0;
    }
    return e;
}

// Text verification needs at least this many symbols left.  With the dense suffix array resolving a row is one load,
// so the text comparison pays off from 4 remaining symbols on (measured on the protein config, 12-symbol queries: 2.58
// -> 1.23 ms per 10 M queries; no effect on 50-symbol DNA queries).  env: GDX_VERIFY_MIN.
inline uint32_t verify_min_remaining(bool dense_sa, const char *env) {
    if (env) return atoi(env) > 0 ? (uint32_t)atoi(env) : 8;
    return dense_sa ? 4 : 8;
}

// The policy travels with the image: the flags and the byte budget come from its header.  Each decision takes the
// bytes the tables built so far take together, the device bytes free right now and the override of the environment
// (GDX_DENSE_SA, GDX_SEED_TABLE, GDX_ROW_CONTEXT: measurements only, read with atoi).
struct AccelPolicy {
    uint64_t n, budget;  // text length, accelerator byte budget (0 = automatic)
    uint32_t ns, lookup_depth;
    bool wide, text;     // 64-bit entries, text section present
    bool no_dense_sa, no_seed_table, no_row_context;

    // the budget minus what is built when a budget is set, else a quarter of the free memory
    uint64_t room(uint64_t used, uint64_t free) const {
        if (budget) return budget > used ? budget - used : 0;
        return free == kFreeUnknown ? 0 : free / 4;
    }

    bool dense_sa(uint64_t used, uint64_t free, const char *env) const {
        if (n == 0) return false;
        if (env) return atoi(env) != 0;
        return !no_dense_sa && n * (wide ? 8ull : 4ull) <= room(used, free);
    }

    // 0: no seed table
    uint32_t seed_depth(uint64_t used, uint64_t free, const char *env) const {
        if (n == 0 || ns < 2) return 0;
        uint32_t depth = 0;
        if (env) {
            depth = atoi(env) > 0 ? (uint32_t)atoi(env) : 0;
        } else {
            if (no_seed_table || free == kFreeUnknown) return 0;
            // the deepest level with at most four entries per text position (then most k-mers of the text have one row
            // and almost no LF step is left): 3.1 Gbp DNA -> depth 16 (34 GB; 0.82 instead of 0.97 ms per 7.5 M queries
            // against depth 15), 500 M residues of protein -> depth 7 (10 GB); the budget below has the last word
            while (seed_entries(ns, depth + 1) && seed_entries(ns, depth + 1) <= 4 * n) ++depth;
            const uint64_t esz = wide ? 16 : 8, r = room(used, free);
            // the finished level must fit the budget; the temporary previous level only has to fit the device
            while (depth > 0 && (seed_entries(ns, depth) * esz > r ||
                                 (seed_entries(ns, depth) + seed_entries(ns, depth - 1)) * esz > free))
                --depth;
        }
        return depth > lookup_depth ? depth : 0;  // the configured table is at least as deep
    }

    bool row_context_possible() const { return n > 0 && !wide && n < (1ull << 32) && ns >= 1 && ns <= 4 && text; }

    // built last (it is the largest: 16 B per text position) and only from what the other two left: the budget when
    // one is set, else up to half of the memory that is still free
    bool row_context(uint64_t used, uint64_t free, const char *env) const {
        if (!row_context_possible()) return false;
        if (env) return atoi(env) != 0;
        return !no_row_context && n * 16 <= (budget ? room(used, free) : 2 * room(used, free));
    }
};

}  // namespace gdx
