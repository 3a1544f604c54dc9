// Host emulation of the device rank-record arithmetic (genedex_b200/csrc/rank_core.h).
// TEST INFRASTRUCTURE: builds the records the way k_pack_k32 / k_pack_kg do, then answers LF and
// symbol_at with the very same __host__ __device__ functions the kernels use, so that the bit-level
// layout can be checked against the oracle on a machine without a GPU.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../genedex_b200/csrc/rank_core.h"

using namespace gdx;

struct Emul {
    RankLayout L;
    uint64_t n;
    uint32_t sigma;
    std::vector<uint8_t> records;
    std::vector<uint64_t> sbc;  // [superblock][noff]
    std::vector<uint64_t> count, border_rows;
};

extern "C" void *emul_build(const uint8_t *bwt, uint64_t n, uint32_t sigma, const uint64_t *count,
                            const uint64_t *border_rows, uint64_t n_border) {
    Emul *e = new Emul();
    e->L = choose_layout(sigma);
    e->n = n;
    e->sigma = sigma;
    e->count.assign(count, count + sigma + 1);
    e->border_rows.assign(border_rows, border_rows + n_border);
    const uint64_t P = 1ull << e->L.log2_pos;
    const uint64_t nrec = (n + 1 + P - 1) / P, nsb = (n + 1 + 65535) / 65536;
    e->records.assign(nrec * e->L.stride, 0);
    e->sbc.assign(nsb * e->L.noff, 0);
    std::vector<uint64_t> run(e->L.noff + 1, 0);  // running #c before the current block within its superblock
    std::vector<uint64_t> total(e->L.noff + 1, 0);
    for (uint32_t c = 1; c <= e->L.noff; ++c) total[c] = count[c];
    for (uint64_t r = 0; r < nrec; ++r) {
        const uint64_t p0 = r * P;
        if ((p0 & 65535) == 0) {
            for (uint32_t c = 1; c <= e->L.noff; ++c) {
                total[c] += run[c];
                run[c] = 0;
                e->sbc[(p0 >> 16) * e->L.noff + (c - 1)] = total[c];
            }
        }
        uint8_t *rec = e->records.data() + r * e->L.stride;
        const uint64_t nsym = p0 >= n ? 0 : (n - p0 < P ? n - p0 : P);
        if (e->L.kind == kLayoutK32) {
            uint64_t w[4] = {0, 0, 0, 0};
            pack_planes64(bwt + p0, (uint32_t)nsym, 3, w);
            for (uint32_t c = 1; c <= e->L.noff; ++c) w[3] |= (run[c] & 0xffff) << (16 * (c - 1));
            memcpy(rec, w, 32);
        } else {
            const uint32_t B = e->L.planes;
            for (uint32_t p = 0; p < B; ++p) {
                uint64_t lo = 0, hi = 0;
                for (uint64_t j = 0; j < nsym; ++j) {
                    uint64_t bit = (uint64_t)((bwt[p0 + j] >> p) & 1u) << (j & 63);
                    if (j < 64) lo |= bit; else hi |= bit;
                }
                memcpy(rec + 16 * p, &lo, 8);
                memcpy(rec + 16 * p + 8, &hi, 8);
            }
            for (uint32_t c = 1; c <= e->L.noff; ++c) {
                uint16_t o = (uint16_t)run[c];
                memcpy(rec + 16 * B + 2 * (c - 1), &o, 2);
            }
        }
        for (uint64_t j = 0; j < nsym; ++j) {
            uint32_t s = bwt[p0 + j];
            if (s >= 1 && s <= e->L.noff) run[s]++;
        }
    }
    return e;
}

extern "C" void emul_free(void *h) { delete (Emul *)h; }

template <int B>
static uint64_t kg_lf(const Emul *e, uint32_t c, uint64_t i) {
    const uint8_t *rec = e->records.data() + (i >> 7) * e->L.stride;
    uint64_t lo[B], hi[B];
    for (int p = 0; p < B; ++p) {
        memcpy(&lo[p], rec + 16 * p, 8);
        memcpy(&hi[p], rec + 16 * p + 8, 8);
    }
    uint16_t off;
    memcpy(&off, rec + 16 * B + 2 * (c - 1), 2);
    return e->sbc[(i >> 16) * e->L.noff + (c - 1)] + off + kg_block_count<B>(lo, hi, c, (uint32_t)(i & 127));
}
template <int B>
static uint32_t kg_sym(const Emul *e, uint64_t i) {
    const uint8_t *rec = e->records.data() + (i >> 7) * e->L.stride;
    uint64_t lo[B], hi[B];
    for (int p = 0; p < B; ++p) {
        memcpy(&lo[p], rec + 16 * p, 8);
        memcpy(&hi[p], rec + 16 * p + 8, 8);
    }
    return kg_symbol_at<B>(lo, hi, (uint32_t)(i & 127));
}

// LF(c, i) = count[c] + rank(c, i), c >= 1  (mirrors lf_pair / K32::lf_derived in kernels.cuh)
extern "C" uint64_t emul_lf(const void *h, uint32_t c, uint64_t i) {
    const Emul *e = (const Emul *)h;
    if (e->L.kind == kLayoutK32) {
        uint64_t w[4];
        memcpy(w, e->records.data() + ((i >> 6) << 5), 32);
        if (c > e->L.noff) {
            uint64_t others = k32_local_rank_sum(w, (uint32_t)(i & 63));
            for (uint32_t s = 1; s <= 4; ++s) others += e->sbc[(i >> 16) * 4 + (s - 1)] - e->count[s];
            uint64_t rank0 = lower_bound_u64(e->border_rows.data(), e->border_rows.size(), i);
            return e->count[5] + (i - rank0 - others);
        }
        return e->sbc[(i >> 16) * e->L.noff + (c - 1)] + k32_local_rank(w, c, (uint32_t)(i & 63));
    }
    switch (e->L.planes) {
    case 1: return kg_lf<1>(e, c, i);
    case 2: return kg_lf<2>(e, c, i);
    case 3: return kg_lf<3>(e, c, i);
    case 4: return kg_lf<4>(e, c, i);
    case 5: return kg_lf<5>(e, c, i);
    case 6: return kg_lf<6>(e, c, i);
    case 7: return kg_lf<7>(e, c, i);
    default: return kg_lf<8>(e, c, i);
    }
}

extern "C" uint32_t emul_symbol_at(const void *h, uint64_t i) {
    const Emul *e = (const Emul *)h;
    if (e->L.kind == kLayoutK32) {
        uint64_t w[4];
        memcpy(w, e->records.data() + ((i >> 6) << 5), 32);
        return k32_symbol_at(w, (uint32_t)(i & 63));
    }
    switch (e->L.planes) {
    case 1: return kg_sym<1>(e, i);
    case 2: return kg_sym<2>(e, i);
    case 3: return kg_sym<3>(e, i);
    case 4: return kg_sym<4>(e, i);
    case 5: return kg_sym<5>(e, i);
    case 6: return kg_sym<6>(e, i);
    case 7: return kg_sym<7>(e, i);
    default: return kg_sym<8>(e, i);
    }
}

extern "C" void emul_layout(const void *h, uint32_t out[6]) {
    const Emul *e = (const Emul *)h;
    out[0] = e->L.kind; out[1] = e->L.planes; out[2] = e->L.noff; out[3] = e->L.stride;
    out[4] = e->L.log2_pos; out[5] = e->L.derived_symbol;
}

// ---- row context table + 2-bit coded queries (genedex_b200/csrc/row_context.h) ------------------------------
#include "../../genedex_b200/csrc/row_context.h"

// entry for SA value `at` over a dense text (one byte per symbol); out = x, y, z, w
extern "C" void emul_ctx_entry(const uint8_t *dense_text, uint64_t at, uint32_t ns, uint32_t *out) {
    const CtxEntry en = ctx_make_entry(at, ns, [&](uint64_t p) { return (uint32_t)dense_text[p]; });
    out[0] = en.x;
    out[1] = en.y;
    out[2] = en.z;
    out[3] = en.w;
}

// the kernel's staging + coding of an IO-byte query: bytes are laid into a 17-word slot at byte offset `mis`
// (garbage everywhere else), coded with codes_from_staged; returns 1 and the 128-bit tail if every byte is a
// searchable symbol, else 0
extern "C" int emul_code_query(const uint8_t *io_to_dense, uint32_t ns, const uint8_t *query, uint32_t tail, uint32_t mis,
                               uint32_t garbage, uint64_t *lo, uint64_t *hi) {
    uint16_t tab2[256];
    for (int b = 0; b < 256; ++b) tab2[b] = ctx_tab2_entry(io_to_dense[b], ns);
    uint32_t slot[17];
    uint8_t *bytes = reinterpret_cast<uint8_t *>(slot);
    for (uint32_t i = 0; i < sizeof slot; ++i) bytes[i] = (uint8_t)(garbage * 2654435761u >> (i % 24));
    memcpy(bytes + mis, query, tail);
    PackedTail t = {0, 0};
    const bool ok = codes_from_staged(tab2, slot, mis, tail, t);
    *lo = t.lo;
    *hi = t.hi;
    return ok ? 1 : 0;
}

extern "C" int emul_ctx_matches(const uint32_t *entry, uint32_t pos, uint64_t ql, uint64_t qh) {
    const CtxEntry en = {entry[0], entry[1], entry[2], entry[3]};
    return ctx_matches(en, pos, ql, qh) ? 1 : 0;
}

extern "C" uint32_t emul_ctx_valid_len(const uint32_t *entry) {
    const CtxEntry en = {entry[0], entry[1], entry[2], entry[3]};
    return ctx_valid_len(en);
}

// the packed kernel's check of a caller's 2-bit codes: 1 if one of the first nsym codes of hi:lo is >= ns
extern "C" int emul_packed_unsearchable(uint64_t lo, uint64_t hi, uint32_t nsym, uint32_t ns) {
    return packed_codes_unsearchable(PackedTail{lo, hi}, nsym, ns) ? 1 : 0;
}
