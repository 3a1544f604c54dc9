// Host build of the chunk schedule of search_host (genedex_b200/csrc/chunk_plan.h) for tests/test_chunk_plan_host.py.
// TEST INFRASTRUCTURE: it drives the schedule the way api.cu does, with packing failures and the hybrid link feedback
// given by the test instead of measured.
#include <cstdint>
#include <vector>

#include "../../genedex_b200/csrc/chunk_plan.h"

// Runs the whole schedule.  limits = {first, max, tail, max_queries}.  At chunk fail_at a chunk that is to be packed
// fails to pack (packing_failed); stage_ms[k] and backlog[k] are what a hybrid run observes after chunk k.  Every chunk
// goes to out as (q0, q1, sym0, sym1, pack, packed); returns the number of chunks, *bad = the query reported for a bad
// boundary (~0 if none), *max_sym = max_chunk_symbols().
extern "C" uint64_t emul_chunk_plan(const uint64_t *offsets, uint64_t fixed_len, uint64_t first_symbol, uint64_t nq,
                                    int prepacked, int pack, int hybrid, const uint64_t *limits, double pack_rate,
                                    double link_bytes_per_ms, int64_t fail_at, const double *stage_ms,
                                    const uint64_t *backlog, uint64_t *out, uint64_t cap, uint64_t *bad,
                                    uint64_t *max_sym) {
    gdx::ChunkPlan plan{offsets, fixed_len, first_symbol, nq, prepacked != 0, pack != 0, hybrid != 0,
                        limits[0], limits[1], limits[2], limits[3], pack_rate, link_bytes_per_ms};
    *bad = ~0ull;
    *max_sym = plan.max_chunk_symbols();
    gdx::Chunk c;
    uint64_t k = 0;
    for (; k < cap && plan.next(c); ++k) {
        if (c.bad_offsets) {
            *bad = c.q0;
            break;
        }
        bool packed = false;
        if (c.nsym() && c.pack) {
            if ((int64_t)k == fail_at) plan.packing_failed();
            else packed = true;
        }
        if (plan.hybrid) plan.after_upload(packed, c.nsym(), stage_ms[k], packed ? backlog[k] : 0);
        const uint64_t row[6] = {c.q0, c.q1, c.sym0, c.sym1, c.pack, packed};
        for (int i = 0; i < 6; ++i) out[6 * k + i] = row[i];
    }
    return k;
}

// gdx::exception_queries into out (room for n entries); returns how many it wrote
extern "C" uint64_t emul_exception_queries(const uint64_t *offsets, uint64_t fixed_len, uint64_t q0, uint64_t q1,
                                           uint64_t sym0, const uint64_t *exc, uint64_t n, uint32_t *out) {
    std::vector<uint32_t> q;
    gdx::exception_queries(offsets, fixed_len, q0, q1, sym0, std::vector<uint64_t>(exc, exc + n), q);
    for (size_t i = 0; i < q.size(); ++i) out[i] = q[i];
    return q.size();
}

// gdx::query_of_symbol
extern "C" uint64_t emul_query_of_symbol(const uint64_t *offsets, uint64_t lo, uint64_t hi, uint64_t sym) {
    return gdx::query_of_symbol(offsets, lo, hi, sym);
}
