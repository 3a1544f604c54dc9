"""GPU tests of the compact seed level (genedex_b200/csrc/compact_seed.h): count and locate queries that start from it
give the oracle's results and the results of the same index without it, the lazy invalid-symbol error stays where the
reference puts it, cursors never use it, and it is built and dropped together with the seed table on every route."""
import os
import random
import tempfile

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(any(v in os.environ for v in ("GDX_DENSE_SA", "GDX_SEED_TABLE", "GDX_ROW_CONTEXT",
                                                      "GDX_VERIFY_MIN", "GDX_FORCE_WIDE")),
                       reason="an environment override replaces the policy (or the entry width) under test"),
]

DEPTH = 4
D = 11  # 4^11 <= 32 n < 4^12 for the ~200 kbp index below; the seed table has depth 9


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    assert genedex_b200._lib.load().gdx_device_count() >= 1
    return genedex_b200


def make_texts():
    """ascii_dna_with_n: N runs, several texts, a repeat-rich text with one 11-mer of more than 2^16 rows"""
    rng = random.Random(17)
    a = bytearray(rng.choice(b"ACGT") for _ in range(90_000))
    for p in range(500, 89_000, 7_001):  # N runs of 1 .. 40 symbols
        a[p:p + 1 + p % 40] = b"N" * len(a[p:p + 1 + p % 40])
    unit = bytes(rng.choice(b"ACGT") for _ in range(300))
    rep = bytearray()
    while len(rep) < 60_000:
        u = bytearray(unit)
        u[rng.randrange(300)] = rng.choice(b"ACGT")  # diverged copies
        rep += u
    return [bytes(a), bytes(rep[:60_000]), b"A" * 70_000, b"ACGTN", b"TTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTT"]


@pytest.fixture(scope="module")
def case(gdx):
    texts = make_texts()
    alph = gdx.alphabet.ascii_dna_with_n()
    oidx = O.OracleIndex.build(texts, O.ALPHABETS["ascii_dna_with_n"](), "u32", sampling_rate=4, lookup_depth=DEPTH)

    def build(budget=0):
        cfg = gdx.FmIndexConfig("u32").suffix_array_sampling_rate(4).lookup_table_depth(DEPTH)
        return cfg.construct_on_device(True, verify=True).accelerator_budget(budget).construct_index(texts, alph)
    pidx = build()
    i = pidx.info()
    assert i.seed_table_depth == 9 and i.compact_seed_depth == D, (i.seed_table_depth, i.compact_seed_depth)
    # a budget that holds the dense suffix array, the seed table and the row context table but not the compact level
    n = i.text_len
    plain = build(n * 4 + 4 ** 9 * 8 + n * 16)
    assert plain.info().compact_seed_depth == 0 and plain.info().row_context_entry_bytes == 16
    return dict(texts=texts, oidx=oidx, pidx=pidx, plain=plain, build=build)


def all_dmers(d):
    codes = np.arange(4 ** d, dtype=np.int64)
    out = np.empty((4 ** d, d), dtype=np.uint8)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    for j in range(d):
        out[:, d - 1 - j] = acgt[(codes >> (2 * j)) & 3]
    return out.reshape(-1)


def check_batch(c, data, off, locate=True):
    oidx, pidx, plain = c["oidx"], c["pidx"], c["plain"]
    want = oidx.count_many_packed(data, off, nthreads=8)
    assert np.array_equal(pidx.count_many_packed(data, off), want)
    assert np.array_equal(plain.count_many_packed(data, off), want)
    if locate:
        ooff, ohits = oidx.locate_many_packed(data, off, nthreads=8)
        for idx in (pidx, plain):
            poff, phits = idx.locate_many_packed(data, off)
            assert np.array_equal(poff, ooff) and np.array_equal(phits, ohits)
    return want


def test_every_dmer_counts_and_locates_like_the_oracle(gdx, case):
    data = all_dmers(D)
    off = np.arange(0, data.size + 1, D, dtype=np.uint64)
    want = check_batch(case, data, off)
    assert want.max() > 1 << 16 and (want >= 3).sum() > 100 and (want == 0).sum() > 0


def test_text_windows_and_random_strings(gdx, case):
    rng = random.Random(3)
    texts = case["texts"]
    qs = []
    for i in range(200_000):
        if i % 2:  # (windows of the all-A text are left to the d-mer test: 70 k hits each)
            t = texts[rng.randrange(2)]
            p = rng.randrange(len(t) - 60)
            q = t[p:p + rng.randrange(1, 60)]
            qs.append(q if b"N" not in q else q.replace(b"N", b"G"))
        else:
            qs.append(bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(0, 30))))
    data, off = O.pack(qs)
    check_batch(case, data, off)
    # fixed-length windows through the host packer (a batch of more than 1 MB) and as a pre-packed batch
    t = texts[1]
    qs = [t[p:p + 24] for p in range(0, len(t) - 24)] * 2
    qs = [q for q in qs if b"N" not in q]
    data, off = O.pack(qs)
    want = check_batch(case, data, off, locate=False)
    packed, first_bad = case["pidx"].pack_queries_2bit(data, off)
    assert first_bad is None
    enc = gdx._lib.GDX_QUERIES_PACKED_2BIT
    assert np.array_equal(case["pidx"].count_many_packed(packed, off, encoding=enc), want)


@pytest.mark.parametrize("bad", [b"!", b"N"])
@pytest.mark.parametrize("where", [D, D - 1, D + 1])
def test_invalid_or_unsearchable_symbol_only_the_compact_level_covers(gdx, case, bad, where):
    """`where` symbols from the end: the compact level covers the 11th and 10th but not the seed table (9)"""
    oidx, pidx, plain = case["oidx"], case["pidx"], case["plain"]
    t = case["texts"][1]
    qs = [t[p:p + 40] for p in range(0, 50_000, 2)]  # > 1 MB: the host packer takes part
    for k in (1000, 7000, 20_000):
        q = bytearray(qs[k])
        q[len(q) - where] = bad[0]
        qs[k] = bytes(q)
    data, off = O.pack(qs)
    try:
        want = oidx.count_many_packed(data, off)
        err = None
    except O.OraclePanic as e:
        want, err = None, e.query
    # the oracle names the first query of the 64-query batch that panics (lib.rs:115), the library the query itself:
    # a window of the text keeps a non-empty interval up to the '!', so the first modified query is the one
    assert (err is not None) == (bad == b"!")
    if err is not None:
        assert err == 1000 // 64 * 64
    for idx in (pidx, plain):
        counts = lambda: idx.count_many_packed(data, off)
        hits_per_query = lambda: np.diff(idx.locate_many_packed(data, off)[0].astype(np.int64))
        for call in (counts, hits_per_query):
            if err is None:
                assert np.array_equal(call().astype(np.int64), want.astype(np.int64))
            else:
                with pytest.raises(gdx.InvalidSymbolError) as ei:
                    call()
                assert ei.value.query == 1000


def test_cursors_do_not_change(gdx, case):
    rng = random.Random(5)
    t = case["texts"][0]
    qs = [t[p:p + rng.randrange(8, 30)].replace(b"N", b"C") for p in (rng.randrange(len(t) - 40) for _ in range(20_000))]
    qs += [bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(11, 20))) for _ in range(20_000)]
    data, off = O.pack(qs)
    os_, oe_ = case["oidx"].cursors_many_packed(data, off)
    for idx in (case["pidx"], case["plain"]):
        ps_, pe_ = idx.cursors_many_packed(data, off)
        assert np.array_equal(os_, ps_) and np.array_equal(oe_, pe_)


def test_every_route_and_the_seed_table_setter(gdx, case):
    pidx = case["pidx"]
    info = pidx.info()
    n = info.text_len
    groups = (4 ** D + 223) // 224
    assert info.compact_seed_bytes >= groups * 64
    with tempfile.TemporaryDirectory() as tmp:
        pidx.save_to_file(os.path.join(tmp, "i.gdx"))
        loaded = gdx.FmIndex.load_from_file(os.path.join(tmp, "i.gdx"))
    from genedex_b200.replicate import ReplicaSet
    rep = ReplicaSet.replicate(pidx, [info.device]).replicas[1]
    for idx in (loaded, rep):
        i = idx.info()
        assert (i.compact_seed_depth, i.compact_seed_bytes) == (D, info.compact_seed_bytes)
    # never without the seed table
    for budget_flags in (dict(seed=False), dict(seed=True)):
        cfg = gdx.FmIndexConfig("u32").suffix_array_sampling_rate(4).lookup_table_depth(DEPTH)
        idx = cfg.seed_table(budget_flags["seed"]).construct_index(case["texts"], gdx.alphabet.ascii_dna_with_n())
        assert idx.info().compact_seed_depth == (D if budget_flags["seed"] else 0)
    # a budget that leaves room for exactly the groups is not enough once the records are counted
    tight = case["build"](n * 4 + 4 ** 9 * 8 + n * 16 + groups * 64)
    assert tight.info().compact_seed_depth in (0, D - 1)
    # dropped with the seed table, rebuilt with it
    rng = random.Random(8)
    t = case["texts"][0]
    data, off = O.pack([t[p:p + 30].replace(b"N", b"A") for p in (rng.randrange(len(t) - 40) for _ in range(5000))])
    want = case["oidx"].count_many_packed(data, off)
    for depth in (0, DEPTH, 9, 10):
        rep.set_seed_table_depth(depth)
        i = rep.info()
        assert i.compact_seed_depth == (D if depth > DEPTH else 0), depth
        assert i.compact_seed_bytes == (info.compact_seed_bytes if depth > DEPTH else 0)
        assert np.array_equal(rep.count_many_packed(data, off), want)
