"""Alphabets whose shape the predefined ones leave out (gdx_testutil.SHAPES), against the CPU oracle.

DNA-like alphabets (at most 4 searchable symbols) with more than 6 dense symbols switch on the host packer, the 2-bit
packed kernel and the row context table on the generic rank layout KG<B>, with 4- or 8-bit text; `acg_n` has 3
searchable symbols on K32; `dna_n_searchable` searches the symbol whose K32 rank is derived (lookup and seed table
fill, extend, 3-bit sort keys).  Every test first asserts the shape it expects, so that a change of the layout choice
cannot move a shape onto another path unnoticed.  The last test covers a caller's pre-packed batch that holds a code
which is not a searchable symbol."""
import ctypes as C
import os
import random
import subprocess
import sys
import zlib

import numpy as np
import pytest

from oracle import oracle as O
import gdx_testutil as util

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = list(util.SHAPES)
SMALL_NS = [s for s in SHAPES if util.oracle_alphabet(s).num_searchable <= 4]
VERIFY_ON = os.environ.get("GDX_VERIFY", "1") != "0"


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    assert genedex_b200._lib.load().gdx_device_count() >= 1
    return genedex_b200


def expect_shape(pidx, name):
    """rank layout, record bytes, text width and row context table as the shape's table row says"""
    _, _, layout, record_bytes, bits = util.SHAPES[name]
    info = pidx.info()
    assert (info.rank_layout, info.rank_record_bytes) == (layout, record_bytes), name
    n = int(info.text_len)
    want = ((n + 1) // 2 if bits == 4 else n) + 16      # (+ 16: one word past the last one, padded to 256 B)
    assert want <= info.text_bytes < want + 256, (name, info.text_bytes, n)
    return info


def symbol_bytes(oa):
    """(IO bytes of searchable symbols, of valid unsearchable ones, invalid bytes)"""
    t = oa.io_to_dense
    return (bytes(b for b in range(256) if 1 <= t[b] <= oa.num_searchable),
            bytes(b for b in range(256) if t[b] > oa.num_searchable),
            bytes(b for b in range(256) if t[b] == 0))


def shape_texts(rng, oa, ntexts, max_len, unsearchable_runs=True):
    """texts over the searchable symbols with runs of 1..60 unsearchable symbols, many of them short"""
    search, unsearch, _ = symbol_bytes(oa)
    texts = []
    for i in range(ntexts):
        m = rng.choice((0, 1, 2, 3, 7, 44, 45, 46, 47, 63, 64, 65, 66, 130)) if i % 3 else rng.randrange(max_len)
        t = bytearray(rng.choice(search) for _ in range(m))
        if unsearchable_runs and unsearch and m > 10:
            for _ in range(rng.randrange(0, 1 + m // 300)):
                p, run = rng.randrange(m), rng.randrange(1, 61)
                t[p:p + run] = bytes(rng.choice(unsearch) for _ in range(len(t[p:p + run])))
        texts.append(bytes(t))
    return texts


LENGTHS = (1, 2, 3, 5, 8, 13, 20, 31, 44, 45, 46, 47, 50, 63, 64, 65, 66, 80, 100, 130)


def edge_queries(rng, oa, texts, n):
    search, _, _ = symbol_bytes(oa)
    nonempty = [t for t in texts if t]
    qs = []
    for _ in range(n):
        m = rng.choice(LENGTHS)
        kind = rng.randrange(6)
        i = rng.randrange(len(nonempty))
        t = nonempty[i]
        p = rng.randrange(len(t))
        q = bytearray(t[p:p + m])
        if kind == 1 and q:            # one substitution
            q[rng.randrange(len(q))] = rng.choice(search)
        elif kind == 2 and i + 1 < len(nonempty):  # glued across the border to the next text
            q = bytearray(t[-rng.randrange(1, m + 1):] + nonempty[i + 1][:rng.randrange(0, m)])
        elif kind == 3:                # reaches over the start of the text
            q = bytearray(rng.choice(search) for _ in range(rng.randrange(1, 4))) + bytearray(t[:m])
        elif kind == 4:                # random string over the searchable symbols
            q = bytearray(rng.choice(search) for _ in range(m))
        qs.append(bytes(q))
    return qs


def check_invalid_per_query(gdx, oidx, pidx, qs):
    """oracle panic <=> InvalidSymbolError, per query and per batched entry point; otherwise the same count"""
    for q in qs:
        try:
            want = int(oidx.count_many([q])[0])
        except O.OraclePanic:
            for fn in (pidx.count_many, pidx.locate_many, pidx.cursors_for_many_queries):
                with pytest.raises(gdx.InvalidSymbolError):
                    fn([q])
            continue
        assert pidx.count_many([q]) == [want], q


EDGE_CONFIGS = [(False, 4, 0), (True, 7, 0), (False, 7, 3), (True, 4, 3)]  # (on_device, sampling rate, depth)


@pytest.mark.parametrize("on_device,s,depth", EDGE_CONFIGS)
@pytest.mark.parametrize("shape", SHAPES)
def test_edges_small_batches(gdx, shape, on_device, s, depth):
    rng = random.Random(zlib.crc32(repr((shape, on_device, s, depth)).encode()))  # (str hashes vary per process)
    oa = util.oracle_alphabet(shape)
    search, unsearch, invalid = symbol_bytes(oa)
    texts = shape_texts(rng, oa, 40, 3000)
    oidx, pidx = util.build_pair(gdx, texts, shape, "u32", s, depth, on_device)
    expect_shape(pidx, shape)
    qs = edge_queries(rng, oa, texts, 1500)
    if depth > 0:  # documented deviation: an unsearchable symbol cannot index the lookup table
        qs = [q for q in qs if not any(b in unsearch for b in q)]
    else:
        qs += [bytes([rng.choice(unsearch)]) * rng.randrange(1, 5) for _ in range(10)] if unsearch else []
    bad = []
    for q in rng.sample(qs, 60):
        if q:
            qb = bytearray(q)
            qb[rng.randrange(len(qb))] = rng.choice(invalid)
            bad.append(bytes(qb))
    small_ns = oa.num_searchable <= 4
    auto_seed = pidx.info().seed_table_depth
    for ctx in ((True, False) if small_ns else (False,)):
        pidx.set_row_context_table(ctx)
        assert pidx.info().row_context_entry_bytes == (16 if ctx else 0)
        for seed in (auto_seed, 0, 5):   # automatic depth, off, explicit
            pidx.set_seed_table_depth(seed)
            assert pidx.info().seed_table_depth == (seed if seed > depth else 0)
            util.assert_same_results(oidx, pidx, qs)
            pidx.count_many(qs)
            if VERIFY_ON:
                assert pidx.stats().verified_queries > 0
            check_invalid_per_query(gdx, oidx, pidx, bad[:30])
    if not small_ns:
        with pytest.raises(gdx.GenedexError):
            pidx.set_row_context_table(True)


def large_case(rng, nrng, oa, n):
    """one text of n symbols (+ two short ones) with unsearchable runs; >= 40 000 windows / random strings / windows
    with a substitution, about 2 % of them holding an unsearchable byte and a few an invalid byte the search never
    reaches.  -> texts, queries, number of queries holding a byte without a 2-bit code"""
    search, unsearch, invalid = symbol_bytes(oa)
    sarr, uarr = np.frombuffer(search, dtype=np.uint8), np.frombuffer(unsearch, dtype=np.uint8)
    text = sarr[nrng.integers(0, sarr.size, n)].copy()
    clean = np.ones(n, dtype=bool)
    for p in nrng.integers(0, n - 60, 200 if uarr.size else 0):
        run = int(nrng.integers(1, 61))
        text[p:p + run] = uarr[nrng.integers(0, uarr.size, run)]
        clean[p:p + run] = False
    texts = [text[:n - 5000].tobytes(), text[n - 5000:n - 4000].tobytes(), text[n - 4000:].tobytes()]
    qs = []
    while len(qs) < 48_000:
        m = rng.choice(LENGTHS[4:] + (30, 40, 90))
        p = rng.randrange(0, n - m)
        kind = rng.randrange(4)
        if kind == 3:
            q = bytes(rng.choice(search) for _ in range(m))
        else:
            if not clean[p:p + m].all() and rng.random() < 0.3:
                continue  # keep the share of exception queries low: the packer then stays on
            q = bytearray(text[p:p + m].tobytes())
            if kind == 2:
                q[rng.randrange(m)] = rng.choice(search)
            q = bytes(q)
        qs.append(q)
    # an invalid byte at the far left of a random (absent) query is never translated (lazy panic of the reference)
    for k in range(40):
        qs[rng.randrange(len(qs))] = bytes([rng.choice(invalid)]) + bytes(rng.choice(search) for _ in range(60))
    n_exc = sum(1 for q in qs if any(b not in search for b in q))
    return texts, qs, n_exc


@pytest.mark.parametrize("shape", SHAPES)
def test_large_batch_packed_kernel(gdx, shape):
    rng = random.Random(31)
    nrng = np.random.default_rng(31)
    oa = util.oracle_alphabet(shape)
    texts, qs, n_exc = large_case(rng, nrng, oa, 1_500_000)
    oidx, pidx = util.build_pair(gdx, texts, shape, "u32", 4, 0)
    expect_shape(pidx, shape)
    data, off = O.pack(qs)
    nq = len(qs)
    assert nq >= 40_000 and data.size > 1 << 20 and n_exc >= 40
    want_s, want_e = oidx.cursors_many_packed(data, off)
    want_o, want_h = oidx.locate_many_packed(data, off)
    small_ns = oa.num_searchable <= 4
    auto_seed = pidx.info().seed_table_depth
    for seed in (auto_seed, 0):      # seed table off: plan_sort sorts the batch
        pidx.set_seed_table_depth(seed)
        for ctx in ((True, False) if small_ns else (False,)):
            pidx.set_row_context_table(ctx)
            assert pidx.info().row_context_entry_bytes == (16 if ctx else 0)
            assert np.array_equal(pidx.count_many_packed(data, off), want_e - want_s)
            st = pidx.stats()
            if small_ns:
                assert st.packed_queries == nq and st.exception_queries == n_exc
            else:
                assert st.packed_queries == 0
            if VERIFY_ON:
                assert st.verified_queries > 0
            gs, ge = pidx.cursors_many_packed(data, off)
            assert np.array_equal(gs, want_s) and np.array_equal(ge, want_e)
            got_o, got_h = pidx.locate_many_packed(data, off)
            assert np.array_equal(got_o, want_o) and np.array_equal(got_h, want_h)
            counts, hits, release = pidx.locate_many_compact_view(data, off)
            try:
                assert np.array_equal(counts.astype(np.uint64), want_o[1:] - want_o[:-1])
                assert np.array_equal(hits.astype(np.uint64), want_h)
            finally:
                release()


def clean_windows(rng, text, search, n, lengths):
    qs = []
    while len(qs) < n:
        m = rng.choice(lengths)
        p = rng.randrange(0, len(text) - m)
        q = bytearray(text[p:p + m])
        if any(b not in search for b in q):
            continue
        if rng.random() < 0.3:
            q[rng.randrange(m)] = rng.choice(search)
        qs.append(bytes(q))
    return qs


def device_run(gdx, pidx, packed, off, m, nq, mode):
    """gdx_count_many_device (mode 1) / gdx_cursors_many_device (mode 0) on a packed batch -> results, error word"""
    import torch
    lib = gdx._lib.load()
    enc = gdx._lib.GDX_QUERIES_PACKED_2BIT
    pad = (-packed.size) % 4
    d_p = torch.from_numpy(np.concatenate([packed, np.zeros(pad, np.uint8)])).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda() if off is not None else None
    d_a = torch.zeros(nq, dtype=torch.int64, device="cuda")
    d_b = torch.zeros(nq, dtype=torch.int64, device="cuda")
    d_err = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    dq = gdx._lib.gdx_queries(d_p.data_ptr(), d_off.data_ptr() if d_off is not None else None, m, nq, enc, 0)
    stream = torch.cuda.current_stream().cuda_stream
    if mode == 1:
        st = lib.gdx_count_many_device(pidx.handle, C.byref(dq), d_a.data_ptr(), d_err.data_ptr(), stream)
    else:
        st = lib.gdx_cursors_many_device(pidx.handle, C.byref(dq), d_a.data_ptr(), d_b.data_ptr(), d_err.data_ptr(), stream)
    assert st == 0
    torch.cuda.synchronize()
    a = d_a.cpu().numpy().astype(np.uint64)
    return (a if mode == 1 else (a, d_b.cpu().numpy().astype(np.uint64))), int(d_err.item())


@pytest.mark.parametrize("shape", SMALL_NS)
def test_prepacked_input(gdx, shape):
    rng = random.Random(8)
    oa = util.oracle_alphabet(shape)
    search, _, _ = symbol_bytes(oa)
    texts = shape_texts(rng, oa, 12, 200_000)
    oidx, pidx = util.build_pair(gdx, texts, shape, "u32", 4, 0)
    expect_shape(pidx, shape)
    enc = gdx._lib.GDX_QUERIES_PACKED_2BIT
    text = max(texts, key=len)
    # variable lengths, many longer than the 64 symbols a query keeps in registers (none shorter than 8: a 1-symbol
    # query has ~10^5 hits to locate)
    qs = clean_windows(rng, text, search, 30_000, LENGTHS[4:])
    data, off = O.pack(qs)
    packed, first_bad = pidx.pack_queries_2bit(data, off)
    assert first_bad is None
    want_s, want_e = oidx.cursors_many_packed(data, off)
    for ctx in (True, False):
        pidx.set_row_context_table(ctx)
        assert np.array_equal(pidx.count_many_packed(packed, off, encoding=enc), want_e - want_s)
        assert pidx.stats().packed_queries == len(qs)
        gs, ge = pidx.cursors_many_packed(packed, off, encoding=enc)
        assert np.array_equal(gs, want_s) and np.array_equal(ge, want_e)
        want_o, want_h = oidx.locate_many_packed(data, off)
        got_o, got_h = pidx.locate_many_packed(packed, off, encoding=enc)
        assert np.array_equal(got_o, want_o) and np.array_equal(got_h, want_h)
        counts, err = device_run(gdx, pidx, packed, off, 0, len(qs), 1)
        assert err == -1 and np.array_equal(counts, want_e - want_s)
        (ds, de), err = device_run(gdx, pidx, packed, off, 0, len(qs), 0)
        assert err == -1 and np.array_equal(ds, want_s) and np.array_equal(de, want_e)
    # fixed odd length: sub-batches do not start on byte boundaries
    m = 67
    fixed = clean_windows(rng, text, search, 20_001, (m,))
    fdata = np.frombuffer(b"".join(fixed), dtype=np.uint8)
    foff = np.arange(len(fixed) + 1, dtype=np.uint64) * m
    fs, fe = oidx.cursors_many_packed(fdata, foff)
    fpacked, first_bad = pidx.pack_queries_2bit(fdata, None, m, len(fixed))
    assert first_bad is None
    assert np.array_equal(pidx.count_many_packed(fpacked, None, m, len(fixed), encoding=enc), fe - fs)
    counts, err = device_run(gdx, pidx, fpacked, None, m, len(fixed), 1)
    assert err == -1 and np.array_equal(counts, fe - fs)
    (ds, de), err = device_run(gdx, pidx, fpacked, None, m, len(fixed), 0)
    assert err == -1 and np.array_equal(ds, fs) and np.array_equal(de, fe)


@pytest.mark.parametrize("shape", SHAPES)
def test_cursors_extend_and_single_queries(gdx, shape):
    rng = random.Random(12)
    oa = util.oracle_alphabet(shape)
    search, unsearch, invalid = symbol_bytes(oa)
    texts = shape_texts(rng, oa, 20, 60_000)
    oidx, pidx = util.build_pair(gdx, texts, shape, "u32", 4, 0, True)
    expect_shape(pidx, shape)
    assert pidx.info().inverse_sample_bytes > 0
    no_isa = (gdx.FmIndexConfig("u32").keep_inverse_samples(False)
              .construct_index(texts, util.product_alphabet(gdx, shape)))
    assert no_isa.info().inverse_sample_bytes == 0
    qs = edge_queries(rng, oa, texts, 3000)
    data, off = O.pack(qs)
    want_s, want_e = oidx.cursors_many_packed(data, off)
    for idx in (pidx, no_isa):
        gs, ge = idx.cursors_many_packed(data, off)
        assert np.array_equal(gs, want_s) and np.array_equal(ge, want_e)
    if VERIFY_ON:
        pidx.cursors_many_packed(data, off)
        assert pidx.stats().verified_queries > 0
    if oa.num_searchable <= 4:  # the CURSORS variant of the packed kernel (isa_row / lf_one)
        clean = [q for q in qs if all(b in search for b in q)]
        cdata, coff = O.pack(clean)
        packed, first_bad = pidx.pack_queries_2bit(cdata, coff)
        assert first_bad is None
        cs, ce = oidx.cursors_many_packed(cdata, coff)
        for idx in (pidx, no_isa):
            gs, ge = idx.cursors_many_packed(packed, coff, encoding=gdx._lib.GDX_QUERIES_PACKED_2BIT)
            assert np.array_equal(gs, cs) and np.array_equal(ge, ce)
    # extend: every valid symbol, unsearchable ones included (the reference ranks them)
    syms = bytes(rng.choice(search + unsearch) for _ in qs)
    es, ee = pidx.extend_many_packed(want_s, want_e, np.frombuffer(syms, dtype=np.uint8))
    for k in range(len(qs)):
        assert (int(es[k]), int(ee[k])) == oidx.extend_query_front((int(want_s[k]), int(want_e[k])), syms[k]), k
    with pytest.raises(gdx.InvalidSymbolError):
        pidx.extend_many_packed(want_s[:3], want_e[:3], np.array([search[0], invalid[0], search[0]], dtype=np.uint8))
    for q in qs[:150]:
        assert pidx.cursor_for_query(q).interval == oidx.cursor_for_query(q), q
    if shape == "dna_n_searchable":  # N is searchable: the seed table ranks the derived symbol
        for d in (1, 2, 5):
            pidx.set_seed_table_depth(d)
            assert pidx.info().seed_table_depth == d
            util.assert_same_results(oidx, pidx, qs + [b"N", b"NN", b"ACGTN" * 9, b"NNNNNNNNNN"])


NEW_SHAPE_SEEDS = 8


@pytest.mark.parametrize("shape", SHAPES)
def test_fuzz_per_shape(shape):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import fuzz_parity
    for seed in range(7_200_000, 7_200_000 + NEW_SHAPE_SEEDS):
        fuzz_parity.one_case(seed, shape)


def test_fuzz_small_ns_shapes_with_every_batch_packed():
    """GDX_PACK_MIN_BYTES=0: the host packer, the packed kernel on KG and the exception re-runs for every batch (the
    switches are read once per process, hence the subprocess)"""
    env = dict(os.environ, GDX_PACK_MIN_BYTES="0", GDX_STAGE_MIN_BYTES="0")
    code = ("import sys; sys.path.insert(0, %r); import fuzz_parity\n"
            "for shape in %r:\n"
            "    for seed in range(7_300_000, 7_300_006): fuzz_parity.one_case(seed, shape)\n"
            "print('ok')" % (os.path.join(ROOT, "tools"), SMALL_NS))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


# ---- a caller's pre-packed batch holding a code that is not a searchable symbol -------------------------------
def poke_code(packed, g, code=3):
    packed[g // 4] = (int(packed[g // 4]) & ~(3 << (2 * (g % 4)))) | (code << (2 * (g % 4)))


M = 100  # query length: 36 symbols in front of the 64 a query keeps in registers
# query positions of the poked code: last symbol (lookup / seed part), LF part, text comparison part, in front of the
# registers
PLACES = {"lookup_or_seed": M - 1, "lf": M - 6, "text_comparison": 40, "before_staged": 5}


@pytest.mark.parametrize("depth", [0, 3])
@pytest.mark.parametrize("shape", ["u8_until_2", "acg_n"])
def test_prepacked_codes_that_are_not_searchable_are_refused(gdx, shape, depth):
    rng = random.Random(77 + depth)
    nrng = np.random.default_rng(77 + depth)
    oa = util.oracle_alphabet(shape)
    assert oa.num_searchable == 3
    search, _, _ = symbol_bytes(oa)
    sarr = np.frombuffer(search, dtype=np.uint8)
    text = sarr[nrng.integers(0, sarr.size, 300_000)].tobytes()
    oidx, pidx = util.build_pair(gdx, [text], shape, "u32", 4, depth)
    enc = gdx._lib.GDX_QUERIES_PACKED_2BIT
    lib = gdx._lib.load()

    def batch(nq):
        qs = [text[p:p + M] for p in (rng.randrange(0, len(text) - M) for _ in range(nq))]
        data = np.frombuffer(b"".join(qs), dtype=np.uint8)
        packed, first_bad = pidx.pack_queries_2bit(data, None, M, nq)
        assert first_bad is None
        return data, packed

    small, small_packed = batch(600)
    big, big_packed = batch(180_000)   # 18 M symbols: more than one chunk of the host pipeline
    want_small = oidx.count_many_packed(small, np.arange(601, dtype=np.uint64) * M)
    want_big = oidx.count_many_packed(big, np.arange(180_001, dtype=np.uint64) * M)
    for seed in ("auto", 0):
        if seed == 0:
            pidx.set_seed_table_depth(0)
        for place, j in PLACES.items():
            for data_packed, nq, first, second in ((small_packed, 600, 200, 400), (big_packed, 180_000, 170_000, 179_999)):
                p = data_packed.copy()
                poke_code(p, second * M + j)
                poke_code(p, first * M + j)
                calls = [lambda: pidx.count_many_packed(p, None, M, nq, encoding=enc)]
                if nq == 600:
                    calls += [lambda: pidx.cursors_many_packed(p, None, M, nq, encoding=enc),
                              lambda: pidx.locate_many_packed(p, None, M, nq, encoding=enc)]
                for call in calls:
                    with pytest.raises(gdx.InvalidSymbolError) as e:
                        call()
                    assert e.value.query == first, (seed, place, nq)
                    assert int(lib.gdx_last_error_query()) == first
                _, err = device_run(gdx, pidx, p, None, M, nq, 1)
                assert err == first, (seed, place, nq)
            # the index is usable afterwards
            assert np.array_equal(pidx.count_many_packed(small_packed, None, M, 600, encoding=enc), want_small)
        assert np.array_equal(pidx.count_many_packed(big_packed, None, M, 180_000, encoding=enc), want_big)
        counts, err = device_run(gdx, pidx, big_packed, None, M, 180_000, 1)
        assert err == -1 and np.array_equal(counts, want_big)
