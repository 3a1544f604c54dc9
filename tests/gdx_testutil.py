"""Shared helpers of the parity tests: the same texts / alphabets / configs for oracle and product."""
import random

import numpy as np

from oracle import oracle as O


def _pairs(letters: bytes):
    return [bytes([c, c + 32]) for c in letters]


# Alphabets built from groups of IO symbols (searchable groups first) and the number of groups that are not
# searchable.  They reach the rank layouts and text widths the library's predefined alphabets leave out: at most
# 4 searchable symbols with more than 6 dense ones (generic layout, packed kernel and row context table all on),
# fewer than 4 searchable symbols on the 32-byte layout, and a searchable symbol whose rank is derived.
SHAPES = {
    # name: (groups, not searchable, rank_layout, rank_record_bytes, text bits)
    "dna_rny": (_pairs(b"ACGTNRY"), 3, 1, 64, 4),                          # sigma 8, KG<3>
    "dna_iupac_kept": (_pairs(b"ACGTNRYKMSWBDHV"), 11, 1, 96, 4),          # sigma 16, KG<4>
    "dna_iupac_gaps": (_pairs(b"ACGTNRYKMSWBDHV") + [b"-", b"*", b"."], 14, 1, 128, 8),  # sigma 19, KG<5>
    "u8_ns4": ([bytes([b]) for b in range(255)], 251, 1, 640, 8),         # sigma 256, KG<8>; byte 255 is invalid
    "acg_n": (_pairs(b"ACGN"), 1, 0, 32, 4),                               # sigma 5, ns 3, K32
    "dna_n_searchable": (_pairs(b"ACGTN"), 0, 0, 32, 4),                   # sigma 6, ns 5: K32 derives the rank of N
}


def product_alphabet(gdx, name):
    A = gdx.alphabet
    if name == "protein20":
        return gdx.Alphabet.from_io_symbols(b"ACDEFGHIKLMNPQRSTVWY", 0)
    if name in SHAPES:
        groups, k = SHAPES[name][:2]
        return gdx.Alphabet.from_ambiguous_io_symbols(groups, k)
    if name.startswith("u8_until_"):
        return A.u8_until(int(name.split("_")[-1]))
    return getattr(A, name)()


def oracle_alphabet(name):
    if name in SHAPES:
        groups, k = SHAPES[name][:2]
        return O.OracleAlphabet(groups, k)
    if name.startswith("u8_until_"):
        return O.u8_until(int(name.split("_")[-1]))
    return O.ALPHABETS[name]()


def searchable_io_symbols(oa):
    """One IO byte per searchable dense symbol."""
    return bytes(oa.dense_to_io[: oa.num_searchable])


def all_io_symbols(oa):
    return bytes(oa.dense_to_io)


def random_texts(rng: random.Random, oa, ntexts, max_len, with_unsearchable=True):
    syms = all_io_symbols(oa) if with_unsearchable else searchable_io_symbols(oa)
    return [bytes(rng.choice(syms) for _ in range(rng.randrange(max_len + 1))) for _ in range(ntexts)]


def random_queries(rng: random.Random, oa, texts, n_sampled, n_random, max_len, searchable_only=False):
    """Windows sampled from the texts plus random strings over the searchable symbols.  With a lookup
    table (depth > 0) a query must not contain a valid-but-unsearchable symbol such as N: the reference
    mis-indexes its table there (lookup_table.rs:154-157), so such windows are dropped on request."""
    syms = searchable_io_symbols(oa)
    ok = set(syms) | {c for c in range(256) if oa.io_to_dense[c] and oa.io_to_dense[c] <= oa.num_searchable}
    qs = []
    nonempty = [t for t in texts if t]
    for _ in range(n_sampled):
        if not nonempty:
            break
        t = rng.choice(nonempty)
        p = rng.randrange(len(t))
        q = t[p:p + rng.randrange(max_len + 1)]
        if searchable_only and any(c not in ok for c in q):
            continue
        qs.append(q)
    for _ in range(n_random):
        qs.append(bytes(rng.choice(syms) for _ in range(rng.randrange(max_len + 1))))
    rng.shuffle(qs)
    return qs


def build_pair(gdx, texts, alph_name, storage="u32", s=4, depth=0, on_device=False):
    oa = oracle_alphabet(alph_name)
    oidx = O.OracleIndex.build(texts, oa, storage, sampling_rate=s, lookup_depth=depth)
    cfg = gdx.FmIndexConfig(storage).suffix_array_sampling_rate(s).lookup_table_depth(depth)
    cfg = cfg.construct_on_device(on_device, verify=on_device)  # the default would be "auto"
    pidx = cfg.construct_index(texts, product_alphabet(gdx, alph_name))
    return oidx, pidx


def assert_same_results(oidx, pidx, queries, check_locate=True):
    data, offsets = O.pack(queries)
    os_, oe_ = oidx.cursors_many_packed(data, offsets)
    ps_, pe_ = pidx.cursors_many_packed(data, offsets)
    assert np.array_equal(os_, ps_) and np.array_equal(oe_, pe_), "intervals differ"
    assert np.array_equal(oidx.count_many_packed(data, offsets), pidx.count_many_packed(data, offsets))
    if check_locate:
        ooff, ohits = oidx.locate_many_packed(data, offsets)
        poff, phits = pidx.locate_many_packed(data, offsets)
        assert np.array_equal(ooff, poff), "hit offsets differ"
        assert np.array_equal(ohits, phits), "hits differ (same SA-row order expected)"
