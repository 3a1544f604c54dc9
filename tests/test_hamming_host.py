"""CPU tests of the Hamming search core (genedex_b200/csrc/hamming.h): the search k_hamming runs, built on the host over
the emulated rank records (tests/host_emul), against a naive scan of every window and the oracle's exact search; the
references of larger indexes (tests/hamming_ref.py) against the naive scan; the core against them on indexes of several
rank superblocks and a homopolymer run.  No GPU compute is called here."""
import ctypes as C
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

from oracle import oracle as O
import gdx_testutil as util
from hamming_ref import (SUPERBLOCK, Cheapest, Naive, Neighbourhood, SeedAndVerify, hamming_queries, hamming_texts,
                         multi_superblock_texts, neighbourhood_size, window_queries)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHABETS = list(util.SHAPES) + ["ascii_dna_with_n", "protein20", "ascii_dna"]


def build_emul(out_dir):
    """tests/host_emul/hamming_emul.cpp as a shared library in out_dir, loaded"""
    out = os.path.join(str(out_dir), "libemul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(ROOT, "tests", "host_emul", "hamming_emul.cpp")])
    lib = C.CDLL(out)
    lib.emul_build.restype = C.c_void_p
    lib.emul_build.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.emul_free.argtypes = [C.c_void_p]
    lib.emul_layout.argtypes = [C.c_void_p, C.c_void_p]
    lib.emul_hamming.restype = C.c_uint64
    lib.emul_hamming.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                 C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return build_emul(tmp_path_factory.mktemp("emul_hamming"))


class EmulIndex:
    """The emulated rank records of an oracle index and the search core over them.  cover adds up, over every search
    run, the counters of emul_hamming: expansions whose borders lie in different superblocks, children of the derived
    symbol past superblock 0, intervals wider than 65 535 rows."""

    def __init__(self, lib, oidx, oa):
        self.lib, self.oa = lib, oa
        self.cover = np.zeros(3, dtype=np.uint64)
        bwt = np.ascontiguousarray(oidx.bwt(), dtype=np.uint8)
        self.n = bwt.size
        freq = np.bincount(bwt, minlength=oa.sigma + 1).astype(np.uint64)
        count = np.zeros(oa.sigma + 1, dtype=np.uint64)
        count[1:] = np.cumsum(freq[: oa.sigma])
        rows = np.flatnonzero(bwt == 0).astype(np.uint64)
        self._keep = (bwt, count, rows if rows.size else np.zeros(1, np.uint64))
        self.h = lib.emul_build(bwt.ctypes.data, self.n, oa.sigma, count.ctypes.data, self._keep[2].ctypes.data,
                                rows.size)

    def layout(self):
        """-> (rank layout: 0 = K32, 1 = KG; derived symbol or 0)"""
        out = (C.c_uint32 * 6)()
        self.lib.emul_layout(self.h, out)
        return out[0], out[5]

    def search(self, query, k):
        qd = np.ascontiguousarray(np.asarray(self.oa.io_to_dense, dtype=np.uint8)[np.frombuffer(query, dtype=np.uint8)])
        buf = qd if qd.size else np.zeros(1, np.uint8)
        occ = np.zeros(k + 1, dtype=np.uint64)
        cap = 1 << 16
        iv = np.zeros(3 * cap, dtype=np.uint64)
        steps = C.c_uint64()
        cover = np.zeros(3, dtype=np.uint64)
        n = self.lib.emul_hamming(self.h, self.oa.num_searchable, self.n, buf.ctypes.data, len(query), k,
                                  occ.ctypes.data, iv.ctypes.data, cap, C.byref(steps), cover.ctypes.data)
        self.cover += cover
        assert n != 2 ** 64 - 1, "pass 2 wrote another number of intervals than pass 1 counted"
        assert n <= cap
        return occ.tolist(), [tuple(int(x) for x in iv[3 * i: 3 * i + 3]) for i in range(n)], steps.value

    def __del__(self):
        self.lib.emul_free(self.h)


@pytest.mark.parametrize("name", ALPHABETS)
def test_hamming_core_equals_naive_scan(emul, name):
    oa = util.oracle_alphabet(name)
    seed = sum(name.encode())
    for trial in range(3):
        rng = random.Random(seed * 10 + trial)
        texts = hamming_texts(rng, oa, rng.randrange(1, 5), 120)
        oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
        naive = Naive(oidx, texts, oa)
        ex = EmulIndex(emul, oidx, oa)
        for k in range(4):
            max_len = 6 if oa.num_searchable > 5 and k >= 2 else 9
            for q in hamming_queries(rng, oa, texts, 25, max_len, k):
                occ, ivs, steps = ex.search(q, k)
                want_occ, want_ivs, _ = naive.expected(q, k)
                assert occ == want_occ, (name, q, k)
                assert ivs == want_ivs, (name, q, k)
                assert [s for s, _, _ in ivs] == sorted(s for s, _, _ in ivs)
                assert all(e > s for s, e, _ in ivs)
                assert all(ivs[i][1] <= ivs[i + 1][0] for i in range(len(ivs) - 1)), "intervals overlap"
                if k == 0 and q:
                    s, e = oidx.cursor_for_query(q)
                    assert ivs == ([(s, e, 0)] if e > s else [])
                assert steps >= (1 if q else 0)


def test_hamming_core_k_at_least_query_length(emul):
    # k >= m: every window of searchable symbols matches; the strata add up to all of them
    oa = util.oracle_alphabet("ascii_dna_with_n")
    rng = random.Random(7)
    texts = hamming_texts(rng, oa, 3, 200, p_other=0.2)
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    naive, ex = Naive(oidx, texts, oa), EmulIndex(emul, oidx, oa)
    for m in range(0, 4):
        q = b"ACGT"[:m]
        occ, ivs, _ = ex.search(q, 3)
        total = sum(len(p) for p in naive.windows(m).values()) if m else oidx.text_len
        assert sum(occ) == total
        assert (occ, ivs) == naive.expected(q, 3)[:2]
        if m:
            assert len(ivs) == len(naive.windows(m))


def test_hamming_core_rows_of_each_interval(emul):
    # the rows of each interval are exactly the occurrences of one window string (locate's input)
    oa = util.oracle_alphabet("dna_n_searchable")
    rng = random.Random(11)
    texts = hamming_texts(rng, oa, 4, 300)
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    naive, ex = Naive(oidx, texts, oa), EmulIndex(emul, oidx, oa)
    sa = oidx.suffix_array()
    for q in hamming_queries(rng, oa, texts, 40, 8, 2):
        _, ivs, _ = ex.search(q, 2)
        _, _, rows = naive.expected(q, 2)
        assert [sorted(sa[s:e].tolist()) for s, e, _ in ivs] == rows


@pytest.mark.parametrize("name", ALPHABETS)
def test_references_equal_naive_scan(name):
    # the two references of larger indexes against the naive scan, on the draws of test_hamming_core_equals_naive_scan
    oa = util.oracle_alphabet(name)
    seed = sum(name.encode())
    checked = [0, 0]
    for trial in range(3):
        rng = random.Random(seed * 10 + trial)
        texts = hamming_texts(rng, oa, rng.randrange(1, 5), 120)
        oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
        naive, nb, sv = Naive(oidx, texts, oa), Neighbourhood(oidx, oa), SeedAndVerify(oidx, oa)
        for k in range(4):
            max_len = 6 if oa.num_searchable > 5 and k >= 2 else 9
            for q in hamming_queries(rng, oa, texts, 25, max_len, k) + [b""]:
                want = naive.expected(q, k)
                if neighbourhood_size(len(q), k, oa.num_searchable) <= 50_000:
                    assert nb.expected(q, k) == want, (name, q, k)
                    checked[0] += 1
                if not q or len(q) >= 3 * (k + 1):
                    assert sv.expected(q, k) == want, (name, q, k)
                    checked[1] += 1
    assert min(checked) >= 30, checked


# (alphabet, symbols, [(k, query lengths)]): k and m per alphabet so that the references stay cheap
LARGE = [
    ("ascii_dna", 400_000, [(1, (8, 15, 30)), (2, (10, 20)), (3, (12, 18, 64, 256))]),
    ("ascii_dna_with_n", 500_000, [(1, (9, 24)), (2, (12, 30)), (3, (12, 16, 100, 255))]),
    ("dna_n_searchable", 300_000, [(1, (7, 20)), (2, (9, 16)), (3, (12, 14, 128))]),
    ("acg_n", 300_000, [(1, (10, 22)), (2, (12,)), (3, (12, 15, 65))]),
    ("dna_rny", 300_000, [(1, (8, 20)), (2, (10,)), (3, (12, 200))]),
    ("protein20", 400_000, [(1, (5, 12)), (2, (9,)), (3, (12, 127, 256))]),
    ("u8_until_40", 300_000, [(1, (4, 10)), (2, (9,)), (3, (12, 64))]),
    ("u8_until_254", 400_000, [(1, (3, 8)), (2, (9,)), (3, (12, 256))]),
]


@pytest.mark.parametrize("name,total,plan", LARGE, ids=[c[0] for c in LARGE])
def test_hamming_core_on_several_superblocks(emul, name, total, plan):
    # the search core against the references on indexes of several rank superblocks (sbc differs from count)
    oa = util.oracle_alphabet(name)
    seed = zlib.crc32(name.encode())
    texts = multi_superblock_texts(seed, oa, total)
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    assert oidx.text_len > 4 * SUPERBLOCK
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    nint = 0
    for k, lengths in plan:
        for m in lengths:
            for q in window_queries(seed + 97 * k + m, oa, texts, 12 if m < 60 else 4, m, k):
                occ, ivs, _ = ex.search(q, k)
                want_occ, want_ivs, _ = ref.expected(q, k)
                assert (occ, ivs) == (want_occ, want_ivs), (name, q, k)
                nint += len(ivs)
    assert nint > 50
    kind, derived = ex.layout()
    if kind == 0:  # K32: expansions across superblocks; children of a searchable derived symbol past superblock 0
        assert ex.cover[0] > 0, ex.cover
        assert (ex.cover[1] > 0) == (0 < derived <= oa.num_searchable), ex.cover


def test_hamming_core_on_a_long_run(emul):
    # A x 70 000 across a superblock boundary: one interval wider than 65 535 rows, u16 in-superblock offsets near
    # their maximum
    oa = util.oracle_alphabet("ascii_dna_with_n")
    nrng = np.random.default_rng(70)
    rand = lambda n: nrng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), n).tobytes()  # noqa: E731
    texts = [rand(40_000), rand(20_000) + b"A" * 70_000 + rand(50_000), b"", rand(30_000)]
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    for m in (1, 2, 12, 20, 100):
        for k in range(4):
            q = b"A" * m
            occ, ivs, _ = ex.search(q, k)
            assert (occ, ivs) == tuple(ref.expected(q, k)[:2]), (m, k)
    assert ex.cover[2] > 0 and ex.cover[0] > 0, ex.cover
