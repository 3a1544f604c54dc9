// genedex_b200.hpp -- header-only C++17 mirror of genedex's public search interface over the C ABI
// (genedex_b200.h).  Same names, argument meaning and error behaviour as the Rust crate
// (src/lib.rs, src/config.rs, src/cursor.rs, src/alphabet.rs); a reference panic is a C++ exception.
// Link with -lgenedex_b200.  All compute runs on the GPU inside the library.
#ifndef GENEDEX_B200_HPP
#define GENEDEX_B200_HPP

#include <cstdint>
#include <cstring>
#include <memory>
#include <set>
#include <stdexcept>
#include <string>
#include <string_view>
#include <tuple>
#include <utility>
#include <vector>

#include "genedex_b200.h"

namespace gdx {

struct Error : std::runtime_error {
    gdx_status status;
    Error(gdx_status s, const std::string &m) : std::runtime_error(m), status(s) {}
};
// the reference panics "symbol in io representation should be valid" (src/alphabet.rs:195-198)
struct InvalidSymbol : Error {
    uint64_t query;
    InvalidSymbol(const std::string &m, uint64_t q) : Error(GDX_ERR_INVALID_SYMBOL, m), query(q) {}
};

inline void check(gdx_status s) {
    if (s == GDX_OK) return;
    if (s == GDX_ERR_INVALID_SYMBOL) throw InvalidSymbol(gdx_last_error_message(), gdx_last_error_query());
    throw Error(s, gdx_last_error_message());
}

// ---- src/alphabet.rs -------------------------------------------------------------------------------
class Alphabet {
public:
    // alphabet.rs:43-75
    static Alphabet from_io_symbols(std::string_view symbols, size_t num_io_symbols_not_searchable = 0) {
        std::vector<std::string> groups;
        for (char c : symbols) groups.emplace_back(1, c);
        return from_ambiguous_io_symbols(groups, num_io_symbols_not_searchable);
    }
    // alphabet.rs:99-149
    static Alphabet from_ambiguous_io_symbols(const std::vector<std::string> &groups,
                                              size_t num_io_symbols_not_searchable = 0) {
        if (groups.empty() || groups.size() > 255)
            throw std::invalid_argument("Alphabet size must be in [1,255] (to leave space for the sentinel).");
        Alphabet a;
        std::memset(a.raw_.io_to_dense, 0, 256);
        std::set<unsigned char> seen;
        for (size_t i = 0; i < groups.size(); ++i) {
            if (groups[i].empty())
                throw std::invalid_argument("Every group of symbols must contain at least one symbol");
            for (unsigned char c : groups[i]) {
                if (!seen.insert(c).second) throw std::invalid_argument("Symbols of the alphabet must be unique.");
                a.raw_.io_to_dense[c] = (uint8_t)(i + 1);
            }
            a.dense_to_io_.push_back(groups[i][0]);
        }
        if (num_io_symbols_not_searchable + 2 > groups.size() + 1)
            throw std::invalid_argument("Invalid alphabet. there must be at least one searchable symbol.");
        a.raw_.num_dense_symbols = (uint32_t)groups.size() + 1;
        a.raw_.num_searchable_dense_symbols = (uint32_t)(groups.size() - num_io_symbols_not_searchable);
        return a;
    }
    uint8_t io_to_dense_representation(uint8_t symbol) const {  // alphabet.rs:195-198
        const uint8_t d = raw_.io_to_dense[symbol];
        if (d == 0) throw std::invalid_argument("symbol in io representation should be valid");
        return d;
    }
    uint8_t dense_to_io_representation(uint8_t symbol) const {  // alphabet.rs:207-210
        if (symbol == 0 || symbol > dense_to_io_.size())
            throw std::invalid_argument("symbol in dense representation should be valid");
        return (uint8_t)dense_to_io_[symbol - 1];
    }
    size_t num_dense_symbols() const { return raw_.num_dense_symbols; }
    size_t num_searchable_dense_symbols() const { return raw_.num_searchable_dense_symbols; }
    const gdx_alphabet &raw() const { return raw_; }

private:
    gdx_alphabet raw_{};
    std::string dense_to_io_;
};

namespace alphabet {  // alphabet.rs:251-345
inline std::vector<std::string> case_pairs(std::string_view upper) {
    std::vector<std::string> g;
    for (char c : upper) g.push_back(std::string{c, (char)(c + 32)});
    return g;
}
inline Alphabet ascii_dna() { return Alphabet::from_ambiguous_io_symbols(case_pairs("ACGT"), 0); }
inline Alphabet ascii_dna_with_n() { return Alphabet::from_ambiguous_io_symbols(case_pairs("ACGTN"), 1); }
inline Alphabet ascii_dna_iupac() { return Alphabet::from_ambiguous_io_symbols(case_pairs("ACGTNRYKMSWBDHV"), 0); }
inline Alphabet ascii_dna_iupac_as_dna_with_n() {
    auto g = case_pairs("ACGT");
    g.push_back("NnRrYyKkMmSsWwBbDdHhVv");
    return Alphabet::from_ambiguous_io_symbols(g, 1);
}
inline Alphabet ascii_amino_acid() { return Alphabet::from_ambiguous_io_symbols(case_pairs("ACDEFGHIKLMNOPQRSTUVWY"), 0); }
inline Alphabet ascii_amino_acid_iupac() {
    auto g = case_pairs("ABCDEFGHIJKLMNOPQRSTUVWXYZ");
    g.push_back("*");
    return Alphabet::from_ambiguous_io_symbols(g, 0);
}
inline Alphabet u8_until(uint8_t max_symbol) {
    std::string s;
    for (int c = 0; c <= max_symbol; ++c) s.push_back((char)c);
    return Alphabet::from_io_symbols(s, 0);
}
inline Alphabet ascii_printable() {
    std::string s;
    for (int c = 32; c < 127; ++c) s.push_back((char)c);
    return Alphabet::from_io_symbols(s, 0);
}
}  // namespace alphabet

// ---- src/lib.rs:331-335 --------------------------------------------------------------------------------
struct Hit {
    size_t text_id;
    size_t position;
    bool operator==(const Hit &o) const { return text_id == o.text_id && position == o.position; }
    bool operator<(const Hit &o) const { return std::tie(text_id, position) < std::tie(o.text_id, o.position); }
};

enum class PerformancePriority : uint32_t { HighSpeed = 0, Balanced = 1, LowMemory = 2 };  // config.rs:89-102
struct I32 { static constexpr uint32_t storage = GDX_I32; };
struct U32 { static constexpr uint32_t storage = GDX_U32; };
struct I64 { static constexpr uint32_t storage = GDX_I64; };

namespace detail {
struct Packed {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> offsets{0};
    template <class Range>
    explicit Packed(const Range &seqs) {
        for (const auto &s : seqs) {
            bytes.insert(bytes.end(), (const uint8_t *)s.data(), (const uint8_t *)s.data() + s.size());
            offsets.push_back(bytes.size());
        }
        if (bytes.empty()) bytes.push_back(0);  // keep a valid pointer
    }
    gdx_queries view() const { return gdx_queries{bytes.data(), offsets.data(), 0, offsets.size() - 1, GDX_QUERIES_IO_BYTES, 0}; }
};
struct Handle {
    gdx_index *p = nullptr;
    ~Handle() { gdx_index_destroy(p); }
};
}  // namespace detail

class Cursor;

// ---- src/lib.rs:93-327 -----------------------------------------------------------------------------------
class FmIndex {
public:
    FmIndex(gdx_index *h, Alphabet a) : h_(std::make_shared<detail::Handle>()), alphabet_(std::move(a)) { h_->p = h; }

    size_t count(std::string_view query) const;                                           // lib.rs:147-149
    template <class Range>
    std::vector<size_t> count_many(const Range &queries) const {                          // lib.rs:155-161
        detail::Packed p(queries);
        std::vector<uint64_t> c(p.offsets.size());
        gdx_queries q = p.view();
        check(gdx_count_many(h_->p, &q, c.data()));
        return std::vector<size_t>(c.begin(), c.end() - 1);
    }
    std::vector<Hit> locate(std::string_view query) const;                                // lib.rs:169-173
    template <class Range>
    std::vector<std::vector<Hit>> locate_many(const Range &queries) const {               // lib.rs:179-185
        detail::Packed p(queries);
        const size_t nq = p.offsets.size() - 1;
        std::vector<uint64_t> off(nq + 1);
        gdx_hit *hits = nullptr;
        uint64_t n = 0;
        gdx_queries q = p.view();
        check(gdx_locate_many(h_->p, &q, off.data(), &hits, &n));
        std::vector<std::vector<Hit>> out(nq);
        for (size_t i = 0; i < nq; ++i)
            for (uint64_t k = off[i]; k < off[i + 1]; ++k) out[i].push_back(Hit{hits[k].text_id, hits[k].position});
        gdx_free_hits(h_->p, hits);
        return out;
    }
    Cursor cursor_empty() const;                                                          // lib.rs:202-210
    Cursor cursor_for_query(std::string_view query) const;                                // lib.rs:217-235
    template <class Range>
    std::vector<Cursor> cursors_for_many_queries(const Range &queries) const;             // lib.rs:241-246

    // approximate search with up to k substitutions (no counterpart in the crate; semantics in genedex_b200.h)
    // [i][d] = occurrences of query i with exactly d mismatches
    template <class Range>
    std::vector<std::vector<size_t>> count_many_hamming(const Range &queries, uint32_t k) const {
        detail::Packed p(queries);
        const size_t nq = p.offsets.size() - 1;
        std::vector<uint64_t> c(nq * (k + 1) + 1);
        gdx_queries q = p.view();
        check(gdx_count_many_hamming(h_->p, &q, k, c.data()));
        std::vector<std::vector<size_t>> out(nq);
        for (size_t i = 0; i < nq; ++i) out[i].assign(c.begin() + i * (k + 1), c.begin() + (i + 1) * (k + 1));
        return out;
    }
    // per query: (interval, mismatches) of every matching window string, sorted by start
    template <class Range>
    std::vector<std::vector<std::pair<Cursor, uint32_t>>> cursors_many_hamming(const Range &queries, uint32_t k) const;
    // per query: the hits of all its intervals in ascending SA-row order
    template <class Range>
    std::vector<std::vector<Hit>> locate_many_hamming(const Range &queries, uint32_t k) const {
        detail::Packed p(queries);
        const size_t nq = p.offsets.size() - 1;
        std::vector<uint64_t> off(nq + 1);
        gdx_hit *hits = nullptr;
        uint64_t n = 0;
        gdx_queries q = p.view();
        check(gdx_locate_many_hamming(h_->p, &q, k, off.data(), &hits, &n));
        std::vector<std::vector<Hit>> out(nq);
        for (size_t i = 0; i < nq; ++i)
            for (uint64_t j = off[i]; j < off[i + 1]; ++j) out[i].push_back(Hit{hits[j].text_id, hits[j].position});
        gdx_free_hits(h_->p, hits);
        return out;
    }

    const Alphabet &alphabet() const { return alphabet_; }                                // lib.rs:283-285
    size_t num_texts() const { return info().num_texts; }                                 // lib.rs:287-289
    size_t total_text_len() const { return info().text_len; }                             // lib.rs:292-294
    gdx_index_info info() const {
        gdx_index_info i{};
        check(gdx_index_get_info(h_->p, &i));
        return i;
    }
    const gdx_index *handle() const { return h_->p; }
    // build (true) or free (false) the dense suffix array accelerator; not while queries are running
    void set_dense_suffix_array(bool on) { check(gdx_index_set_dense_suffix_array(h_->p, on ? 1 : 0)); }
    // (re)build the seed table accelerator at this depth, 0 frees it; not while queries are running
    void set_seed_table_depth(int depth) { check(gdx_index_set_seed_table_depth(h_->p, depth)); }
    // build (true) or free (false) the row context table accelerator; not while queries are running
    void set_row_context_table(bool on) { check(gdx_index_set_row_context_table(h_->p, on ? 1 : 0)); }

private:
    std::shared_ptr<detail::Handle> h_;  // FmIndex: Clone (lib.rs:92) shares the device image
    Alphabet alphabet_;
};

// ---- src/cursor.rs:16-73 ---------------------------------------------------------------------------------
class Cursor {
public:
    Cursor(const FmIndex *index, uint64_t start, uint64_t end) : index_(index), start_(start), end_(end) {}
    void extend_query_front(uint8_t symbol) {  // cursor.rs:34-38
        check(gdx_extend_many(index_->handle(), &start_, &end_, &symbol, 1));
    }
    size_t count() const { return end_ - start_; }  // cursor.rs:61-63
    std::vector<Hit> locate() const {               // cursor.rs:71-73
        uint64_t off[2];
        gdx_hit *hits = nullptr;
        uint64_t n = 0;
        check(gdx_locate_intervals(index_->handle(), &start_, &end_, 1, off, &hits, &n));
        std::vector<Hit> out;
        for (uint64_t k = 0; k < n; ++k) out.push_back(Hit{hits[k].text_id, hits[k].position});
        gdx_free_hits(index_->handle(), hits);
        return out;
    }
    std::pair<uint64_t, uint64_t> interval() const { return {start_, end_}; }

private:
    const FmIndex *index_;
    uint64_t start_, end_;
};

inline Cursor FmIndex::cursor_empty() const { return Cursor(this, 0, total_text_len()); }
inline Cursor FmIndex::cursor_for_query(std::string_view query) const {
    uint64_t s = 0, e = 0;
    check(gdx_cursor_for_query(h_->p, (const uint8_t *)query.data(), query.size(), &s, &e));
    return Cursor(this, s, e);
}
inline size_t FmIndex::count(std::string_view query) const { return cursor_for_query(query).count(); }
inline std::vector<Hit> FmIndex::locate(std::string_view query) const { return cursor_for_query(query).locate(); }
template <class Range>
std::vector<Cursor> FmIndex::cursors_for_many_queries(const Range &queries) const {
    detail::Packed p(queries);
    const size_t nq = p.offsets.size() - 1;
    std::vector<uint64_t> s(nq + 1), e(nq + 1);
    gdx_queries q = p.view();
    check(gdx_cursors_many(h_->p, &q, s.data(), e.data()));
    std::vector<Cursor> out;
    for (size_t i = 0; i < nq; ++i) out.emplace_back(this, s[i], e[i]);
    return out;
}
template <class Range>
std::vector<std::vector<std::pair<Cursor, uint32_t>>> FmIndex::cursors_many_hamming(const Range &queries, uint32_t k) const {
    detail::Packed p(queries);
    const size_t nq = p.offsets.size() - 1;
    std::vector<uint64_t> off(nq + 1);
    gdx_hamming_interval *iv = nullptr;
    uint64_t n = 0;
    gdx_queries q = p.view();
    check(gdx_cursors_many_hamming(h_->p, &q, k, off.data(), &iv, &n));
    std::vector<std::vector<std::pair<Cursor, uint32_t>>> out(nq);
    for (size_t i = 0; i < nq; ++i)
        for (uint64_t j = off[i]; j < off[i + 1]; ++j) out[i].emplace_back(Cursor(this, iv[j].start, iv[j].end), iv[j].mismatches);
    gdx_free_hits(h_->p, (gdx_hit *)iv);
    return out;
}

// ---- one batch over several GPUs (no counterpart in the crate; SURVEY 8e) ---------------------------------
// Full replicas of an index on other devices (one ncclBroadcast of the device image) and the *_many calls over
// all of them: the batch is cut into contiguous ranges by the library, results come back in input order.
class ReplicaSet {
public:
    ReplicaSet(const FmIndex &index, const std::vector<int32_t> &other_devices) {
        std::vector<gdx_index *> out(other_devices.size(), nullptr);
        check(gdx_index_replicate(index.handle(), other_devices.data(), (int32_t)other_devices.size(), out.data()));
        replicas_.push_back(index);
        for (gdx_index *h : out) replicas_.emplace_back(h, index.alphabet());
        for (const FmIndex &r : replicas_) handles_.push_back(const_cast<gdx_index *>(r.handle()));
    }
    size_t size() const { return replicas_.size(); }
    template <class Range>
    std::vector<size_t> count_many(const Range &queries) const {                          // lib.rs:155-161
        detail::Packed p(queries);
        std::vector<uint64_t> c(p.offsets.size());
        gdx_queries q = p.view();
        check(gdx_count_many_sharded(handles_.data(), (uint32_t)handles_.size(), 0, (uint32_t)handles_.size(), &q, c.data()));
        return std::vector<size_t>(c.begin(), c.end() - 1);
    }
    template <class Range>
    std::vector<std::vector<Hit>> locate_many(const Range &queries) const {               // lib.rs:179-185
        detail::Packed p(queries);
        const size_t nq = p.offsets.size() - 1, ns = handles_.size();
        std::vector<uint64_t> off(nq + 1), first(ns + 1);
        std::vector<gdx_hit *> hits(ns, nullptr);
        gdx_queries q = p.view();
        check(gdx_locate_many_sharded(handles_.data(), (uint32_t)ns, 0, (uint32_t)ns, &q, off.data(), hits.data(), first.data()));
        std::vector<std::vector<Hit>> out(nq);
        for (size_t k = 0; k < ns; ++k) {
            uint64_t b = 0, e = 0;
            gdx_shard_range(nq, (uint32_t)k, (uint32_t)ns, &b, &e);
            for (uint64_t i = b; i < e; ++i)
                for (uint64_t j = off[i]; j < off[i + 1]; ++j)
                    out[i].push_back(Hit{hits[k][j - first[k]].text_id, hits[k][j - first[k]].position});
            gdx_free_hits(handles_[k], hits[k]);
        }
        return out;
    }

private:
    std::vector<FmIndex> replicas_;
    std::vector<gdx_index *> handles_;
};

// ---- src/config.rs:9-82 ---------------------------------------------------------------------------------
template <class I = I32>
class FmIndexConfig {
public:
    FmIndexConfig &suffix_array_sampling_rate(uint32_t rate) {
        if (rate == 0) throw std::invalid_argument("suffix_array_sampling_rate > 0");  // config.rs:28
        cfg_.suffix_array_sampling_rate = rate;
        return *this;
    }
    FmIndexConfig &lookup_table_depth(uint32_t depth) {
        cfg_.lookup_table_depth = depth;
        return *this;
    }
    FmIndexConfig &construction_performance_priority(PerformancePriority p) {
        cfg_.performance_priority = (uint32_t)p;
        return *this;
    }
    // additions of this engine
    FmIndexConfig &construct_on_device(bool on = true, bool verify = false) {
        cfg_.construction = on ? GDX_CONSTRUCT_DEVICE : GDX_CONSTRUCT_HOST;
        cfg_.flags = (cfg_.flags & ~GDX_FLAG_VERIFY_SUFFIX_ARRAY) | (verify ? GDX_FLAG_VERIFY_SUFFIX_ARRAY : 0);
        return *this;
    }
    FmIndexConfig &keep_text(bool keep = true) { return flag(GDX_FLAG_NO_TEXT, !keep); }
    FmIndexConfig &keep_inverse_samples(bool keep = true) { return flag(GDX_FLAG_NO_INVERSE_SAMPLES, !keep); }
    // dense suffix array accelerator (gdx_index_set_dense_suffix_array): default = built when memory is ample
    FmIndexConfig &dense_suffix_array(bool allow = true) { return flag(GDX_FLAG_NO_DENSE_SUFFIX_ARRAY, !allow); }
    // seed table accelerator (gdx_index_set_seed_table_depth): default = built when memory is ample
    FmIndexConfig &seed_table(bool allow = true) { return flag(GDX_FLAG_NO_SEED_TABLE, !allow); }
    // row context table accelerator (gdx_index_set_row_context_table): default = built when memory is ample
    FmIndexConfig &row_context_table(bool allow = true) { return flag(GDX_FLAG_NO_ROW_CONTEXT_TABLE, !allow); }
    FmIndexConfig &device(int ordinal) {
        cfg_.device = ordinal;
        return *this;
    }
    template <class Range>
    FmIndex construct_index(const Range &texts, const Alphabet &alphabet) const {  // config.rs:63-69
        detail::Packed p(texts);
        gdx_index *h = nullptr;
        check(gdx_index_build(p.bytes.data(), p.offsets.data(), p.offsets.size() - 1, &alphabet.raw(), &cfg_, &h));
        return FmIndex(h, alphabet);
    }

private:
    FmIndexConfig &flag(uint32_t bit, bool on) {
        cfg_.flags = on ? (cfg_.flags | bit) : (cfg_.flags & ~bit);
        return *this;
    }
    // config.rs:72-82 defaults: sampling rate 4, lookup depth 0, Balanced
    gdx_config cfg_{I::storage, 4, 0, (uint32_t)PerformancePriority::Balanced, GDX_CONSTRUCT_AUTO, -1, 0, 0};
};

}  // namespace gdx
#endif
