"""The accelerator policy on the device (include/genedex_b200.h, DESIGN.md "Accelerator policy"): every way of creating
an index builds the tables a small model of the documented policy predicts, and dropping and rebuilding tables leaves an
index that behaves like a freshly built one with the same tables."""
import ctypes as C
import os
import random
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
import gdx_testutil as util

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(any(v in os.environ for v in ("GDX_DENSE_SA", "GDX_SEED_TABLE", "GDX_ROW_CONTEXT",
                                                      "GDX_VERIFY_MIN", "GDX_FORCE_WIDE")),
                       reason="an environment override replaces the policy (or the entry width) under test"),
]

ALPH, STORAGE, RATE, DEPTH = "ascii_dna", "u32", 4, 2
NS = 4  # searchable symbols of ascii_dna
NO_DENSE_SA, NO_SEED_TABLE, NO_ROW_CONTEXT = 8, 16, 32  # GDX_FLAG_NO_*


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    assert genedex_b200._lib.load().gdx_device_count() >= 1
    return genedex_b200


@pytest.fixture(scope="module")
def corpus():
    rng = random.Random(41)
    texts = [bytes(rng.choice(b"ACGT") for _ in range(k)) for k in (25_000, 10_000, 4_997)]
    oidx = O.OracleIndex.build(texts, util.oracle_alphabet(ALPH), STORAGE, sampling_rate=RATE, lookup_depth=DEPTH)
    return texts, oidx


def model(n, flags, budget, text):
    """(dense_suffix_array_bytes, seed_table_depth, seed_table_bytes, row_context_entry_bytes) of the documented policy
    for 32-bit entries, with device memory far larger than these tables when no budget is set"""
    room = (lambda used: max(budget - used, 0)) if budget else (lambda used: 1 << 62)
    dense = n * 4 if not flags & NO_DENSE_SA and n * 4 <= room(0) else 0
    depth, seed = 0, 0
    if not flags & NO_SEED_TABLE:
        depth = max(d for d in range(40) if NS ** d <= 4 * n)
        while depth > 0 and NS ** depth * 8 > room(dense):
            depth -= 1
        depth = depth if depth > DEPTH else 0
        seed = NS ** depth * 8 if depth else 0
    row = 16 if text and not flags & NO_ROW_CONTEXT and n * 16 <= room(dense + seed) else 0
    return dense, depth, seed, row


def accel(idx):
    i = idx.info()
    return i.dense_suffix_array_bytes, i.seed_table_depth, i.seed_table_bytes, i.row_context_entry_bytes


def routes(gdx, corpus, flags, budget):
    """(name, index, has text section) for every way of creating an index, all under the same policy"""
    import torch
    texts, oidx = corpus
    lib = gdx._lib.load()
    alphabet = util.product_alphabet(gdx, ALPH)

    def construct(on_device):
        cfg = gdx.FmIndexConfig(STORAGE).suffix_array_sampling_rate(RATE).lookup_table_depth(DEPTH)
        cfg = cfg.construct_on_device(on_device).accelerator_budget(budget)
        cfg = cfg.dense_suffix_array(not flags & NO_DENSE_SA).seed_table(not flags & NO_SEED_TABLE)
        return cfg.row_context_table(not flags & NO_ROW_CONTEXT).construct_index(texts, alphabet)

    host = construct(False)
    yield "host construction", host, True
    yield "device construction", construct(True), True
    parts, _keep = util.reference_parts(gdx, oidx, util.oracle_alphabet(ALPH), RATE, DEPTH)
    parts.flags, parts.accelerator_budget_bytes = flags, budget
    h = C.c_void_p()
    assert lib.gdx_index_create_from_bwt(oidx.bwt().ctypes.data, C.byref(parts), -1, C.byref(h)) == 0
    yield "create_from_bwt", gdx.FmIndex(h, alphabet), False
    h = C.c_void_p()
    assert lib.gdx_index_create_from_parts(C.byref(parts), -1, C.byref(h)) == 0
    yield "create_from_parts", gdx.FmIndex(h, alphabet), False
    with tempfile.TemporaryDirectory() as tmp:
        host.save_to_file(os.path.join(tmp, "index.gdx"))
        loaded = gdx.FmIndex.load_from_file(os.path.join(tmp, "index.gdx"))
    yield "save + load", loaded, True
    hdr = (C.c_uint8 * lib.gdx_index_header_bytes())()
    img, nbytes = C.c_void_p(), C.c_uint64()
    assert lib.gdx_index_export(host.handle, hdr, C.byref(img), C.byref(nbytes)) == 0

    class _View:  # zero-copy torch view of the exported image
        __cuda_array_interface__ = {"shape": (nbytes.value,), "typestr": "|u1", "data": (img.value, False),
                                    "version": 2}

    mem = torch.as_tensor(_View(), device="cuda").clone()
    torch.cuda.synchronize()
    h = C.c_void_p()
    assert lib.gdx_index_adopt_image(hdr, mem.data_ptr(), -1, 0, C.byref(h)) == 0
    yield "export + adopt", gdx.FmIndex(h, alphabet, keepalive=mem), True
    outs = (C.c_void_p * 1)()
    assert lib.gdx_index_replicate(host.handle, (C.c_int32 * 1)(host.info().device), 1, outs) == 0
    yield "replicate", gdx.FmIndex(C.c_void_p(outs[0]), alphabet), True


def budgets(n):
    seed_auto = max(d for d in range(40) if NS ** d <= 4 * n)
    return {
        "automatic": 0,
        "nothing fits": 100,
        "only the dense suffix array": n * 4 + 500,
        "a shallower seed table": n * 4 + NS ** (seed_auto - 2) * 8 + 10,
        "no room left for the row context": n * 4 + NS ** seed_auto * 8 + n * 16 - 1,
        "all three": n * 4 + NS ** seed_auto * 8 + n * 16,
    }


def check_routes(gdx, corpus, flags, budget):
    n = corpus[1].text_len
    for name, idx, text in routes(gdx, corpus, flags, budget):
        assert idx.info().text_len == n
        assert accel(idx) == model(n, flags, budget, text), (name, flags, budget)


@pytest.mark.parametrize("case", ["automatic", "nothing fits", "only the dense suffix array", "a shallower seed table",
                                  "no room left for the row context", "all three"])
def test_every_route_builds_what_the_budget_allows(gdx, corpus, case):
    n = corpus[1].text_len
    budget = budgets(n)[case]
    want = model(n, 0, budget, True)
    expected = {"automatic": lambda w: all(w), "nothing fits": lambda w: not any(w),
                "only the dense suffix array": lambda w: w[0] and not w[1] and not w[3],
                "a shallower seed table": lambda w: w[0] and 0 < w[1] < model(n, 0, 0, True)[1] and not w[3],
                "no room left for the row context": lambda w: w[0] and w[1] == model(n, 0, 0, True)[1] and not w[3],
                "all three": lambda w: all(w)}[case]
    assert expected(want), want  # the budget exercises the case it is named for
    check_routes(gdx, corpus, 0, budget)


@pytest.mark.parametrize("flag", [NO_DENSE_SA, NO_SEED_TABLE, NO_ROW_CONTEXT])
@pytest.mark.parametrize("case", ["automatic", "all three"])
def test_every_route_honours_the_flags(gdx, corpus, flag, case):
    check_routes(gdx, corpus, flag, budgets(corpus[1].text_len)[case])


def fixed_batch(texts):
    rng = random.Random(5)
    qs = []
    for i in range(3000):
        t = texts[rng.randrange(len(texts))]
        p = rng.randrange(len(t) - 70)
        qs.append(t[p:p + rng.choice([6, 9, 12, 16, 24, 40, 64])] if i % 3 else
                  bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(0, 30))))
    return O.pack(qs)


def observe(idx, oidx, data, offsets):
    """accelerator fields, and the verified queries of counting the batch; results are checked against the oracle"""
    some = [bytes(data[offsets[i]:offsets[i + 1]]) for i in range(0, len(offsets) - 1, 7)]
    util.assert_same_results(oidx, idx, some)
    assert np.array_equal(idx.count_many_packed(data, offsets), oidx.count_many_packed(data, offsets))
    return accel(idx), idx.stats().verified_queries


def test_dropping_and_rebuilding_tables_matches_a_fresh_index(gdx, corpus):
    texts, oidx = corpus
    data, offsets = fixed_batch(texts)
    alphabet = util.product_alphabet(gdx, ALPH)
    fresh = {}
    for dense in (False, True):
        for seed in (False, True):
            for row in (False, True):
                cfg = gdx.FmIndexConfig(STORAGE).suffix_array_sampling_rate(RATE).lookup_table_depth(DEPTH)
                cfg = cfg.dense_suffix_array(dense).seed_table(seed).row_context_table(row)
                fresh[(dense, seed, row)] = observe(cfg.construct_index(texts, alphabet), oidx, data, offsets)
    assert fresh[(True, False, False)][1] != fresh[(False, False, False)][1]  # the threshold of the dense SA shows
    depth = fresh[(True, True, True)][0][1]
    assert depth > DEPTH

    def apply(idx, state, op):
        kind, on = op
        if kind == "dense":
            idx.set_dense_suffix_array(on)
            return (on, state[1], state[2])
        if kind == "seed":
            idx.set_seed_table_depth(depth if on else DEPTH)  # a depth not above the configured one drops the table
            return (state[0], on, state[2])
        idx.set_row_context_table(on)
        return (state[0], state[1], on)

    orders = [
        [("dense", 0), ("seed", 0), ("row", 0), ("row", 1), ("dense", 1), ("seed", 1)],
        [("row", 0), ("dense", 0), ("dense", 1), ("dense", 1), ("seed", 0), ("row", 1), ("seed", 1)],
        [("seed", 0), ("seed", 1), ("seed", 1), ("dense", 0), ("row", 0), ("seed", 0), ("dense", 1), ("row", 1)],
    ]
    for order in orders:
        idx = gdx.FmIndexConfig(STORAGE).suffix_array_sampling_rate(RATE).lookup_table_depth(DEPTH).construct_index(
            texts, alphabet)
        state = (True, True, True)
        assert observe(idx, oidx, data, offsets) == fresh[state]
        for op in order:
            state = apply(idx, state, op)
            assert observe(idx, oidx, data, offsets) == fresh[state], (order, op)
