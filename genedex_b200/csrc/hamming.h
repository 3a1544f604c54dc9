// hamming.h -- backtracking backward search with up to k substitutions (gdx_*_many_hamming).
//
// Semantics (include/genedex_b200.h, "approximate search"):
//   - a query of length m matches at text position p with d mismatches when the window [p, p + m) lies inside one
//     text, every symbol of it is a searchable dense symbol (1..ns), and it differs from the query (compared in the
//     dense representation) in exactly d <= k positions.  A window holding `N`, another non-searchable symbol or a
//     sentinel never matches;
//   - every distinct matching window string is one non-empty SA interval [start, end); its mismatch count is its
//     Hamming distance to the query.  The intervals of a query are pairwise disjoint and are returned sorted by start;
//   - k = 0 gives the interval of the exact search (none when it is empty); the empty query gives [0, n) with 0
//     mismatches.
//
// The search is a depth-first walk of the backward-search trie from [0, n).  A node at query position pos (the
// symbols pos..m-1 are consumed) with d mismatches has one child per searchable symbol c: the interval
// [LF(c, start), LF(c, end)), which costs a mismatch unless c is the query symbol at pos - 1.  Empty children and
// children over the budget are pruned.  Once a node has used the whole budget the rest of the query is an exact
// backward search that keeps no frame, so the frames on the stack always belong to the consecutive query positions
// m, m - 1, ...: the stack holds at most m <= kHammingMaxQueryLen frames, whatever the number of results.
// The leaves do not come out in SA order: an extension to the left moves to the block of its first symbol, away from
// its parent's interval.  Pass 2 therefore writes every interval as the pair (start, (end - start) << 2 | d) and a
// per-query sort by start (api.cu) gives the canonical order; the intervals are disjoint, so the starts are distinct.
//
// The rank source R is what differs between the device layouts and the host emulation (tests/host_emul):
//   R::Node                                  what one expansion keeps of a node (its children, or just its interval)
//   R::ns, R::n                              searchable symbols, text length
//   expand(s, e, Node &)                     one node expansion (s < e)
//   child(const Node &, c, s &, e &)         interval of child c of an expanded node
//   step(c, s &, e &)                        one exact LF pair (c: the query symbol)
// Everything here is __host__ __device__ (GDX_HD, rank_core.h).
#ifndef GDX_HAMMING_H
#define GDX_HAMMING_H

#include <stdint.h>

#include "rank_core.h"

namespace gdx {

constexpr uint32_t kHammingMaxMismatches = 3;  // GDX_HAMMING_MAX_MISMATCHES
constexpr uint32_t kHammingMaxQueryLen = 256;  // GDX_HAMMING_MAX_QUERY_LEN

// one interval of the result (the layout of gdx_hamming_interval)
struct HammingInterval {
    uint64_t start, end;
    uint32_t mismatches, reserved;
};

template <class Node>
struct HammingFrame {
    Node node;      // the expanded node
    uint32_t d;     // its mismatches
    uint32_t next;  // next child symbol to try
};

// Runs the search of one query; sym(j) = dense symbol of query position j (1..ns, checked by the caller).
// emit(start, end, d) is called once per matching interval.  `stack` holds m frames.
// Returns the number of node expansions (an expansion of a node with a budget left, or one exact LF pair).
#if defined(__CUDACC__)
#pragma nv_exec_check_disable  // the device rank sources are __device__ only
#endif
template <class R, class Q, class Emit>
GDX_HD uint64_t hamming_search(const R &rs, const Q &sym, uint32_t m, uint32_t k,
                               HammingFrame<typename R::Node> *stack, Emit &emit) {
    uint64_t expansions = 0;
    int top = -1;  // stack[t] is the node at query position m - t
    uint64_t s = 0, e = rs.n;
    uint32_t d = 0, pos = m;
    for (;;) {
        // enter the node (s, e) at query position pos with d mismatches (s < e)
        if (pos == 0) {
            emit(s, e, d);
        } else if (d == k) {  // no budget left: the rest is an exact backward search
            while (pos > 0 && s != e) {
                rs.step(sym(pos - 1), s, e);
                --pos;
                ++expansions;
            }
            if (s != e) emit(s, e, d);
        } else {
            ++top;
            rs.expand(s, e, stack[top].node);
            stack[top].d = d;
            stack[top].next = 1;
            ++expansions;
        }
        // the next child to enter: the deepest frame with one left
        bool found = false;
        while (top >= 0 && !found) {
            HammingFrame<typename R::Node> &f = stack[top];
            const uint32_t p = m - (uint32_t)top;
            const uint32_t qc = sym(p - 1);
            while (f.next <= rs.ns) {
                const uint32_t c = f.next++;
                const uint32_t dc = f.d + (c != qc ? 1u : 0u);
                if (dc > k) continue;
                uint64_t cs, ce;
                rs.child(f.node, c, cs, ce);
                if (cs == ce) continue;
                s = cs;
                e = ce;
                d = dc;
                pos = p - 1;
                found = true;
                break;
            }
            if (!found) --top;
        }
        if (!found) break;
    }
    return expansions;
}

// pass 1: per-stratum occurrences and number of intervals
struct HammingCounter {
    uint64_t occ[kHammingMaxMismatches + 1] = {0, 0, 0, 0};
    uint64_t intervals = 0;
    GDX_HD void operator()(uint64_t s, uint64_t e, uint32_t d) {
        occ[d] += e - s;
        ++intervals;
    }
};

// pass 2: the intervals of a query from its CSR offset on, in search order, as sort key (start) and value
// ((end - start) << 2 | d)
struct HammingWriter {
    uint64_t *keys, *vals;
    uint64_t at;
    GDX_HD void operator()(uint64_t s, uint64_t e, uint32_t d) {
        keys[at] = s;
        vals[at] = ((e - s) << 2) | d;
        ++at;
    }
};
GDX_HD HammingInterval hamming_decode(uint64_t key, uint64_t val) {
    HammingInterval h;
    h.start = key;
    h.end = key + (val >> 2);
    h.mismatches = (uint32_t)(val & 3u);
    h.reserved = 0;
    return h;
}

}  // namespace gdx
#endif
