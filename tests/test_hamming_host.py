"""CPU tests of the Hamming search core (genedex_b200/csrc/hamming.h): the search k_hamming runs, built on the host over
the emulated rank records (tests/host_emul), against a naive scan of every window and the oracle's exact search.
No GPU compute is called here."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
import gdx_testutil as util
from hamming_ref import Naive, hamming_queries, hamming_texts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHABETS = list(util.SHAPES) + ["ascii_dna_with_n", "protein20", "ascii_dna"]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    out = tmp_path_factory.mktemp("emul_hamming") / "libemul.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(ROOT, "tests", "host_emul", "hamming_emul.cpp")])
    lib = C.CDLL(str(out))
    lib.emul_build.restype = C.c_void_p
    lib.emul_build.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.emul_free.argtypes = [C.c_void_p]
    lib.emul_hamming.restype = C.c_uint64
    lib.emul_hamming.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                 C.c_void_p, C.c_uint64, C.c_void_p]
    return lib


class EmulIndex:
    def __init__(self, lib, oidx, oa):
        self.lib, self.oa = lib, oa
        bwt = np.ascontiguousarray(oidx.bwt(), dtype=np.uint8)
        self.n = bwt.size
        freq = np.bincount(bwt, minlength=oa.sigma + 1).astype(np.uint64)
        count = np.zeros(oa.sigma + 1, dtype=np.uint64)
        count[1:] = np.cumsum(freq[: oa.sigma])
        rows = np.flatnonzero(bwt == 0).astype(np.uint64)
        self._keep = (bwt, count, rows if rows.size else np.zeros(1, np.uint64))
        self.h = lib.emul_build(bwt.ctypes.data, self.n, oa.sigma, count.ctypes.data, self._keep[2].ctypes.data,
                                rows.size)

    def search(self, query, k):
        qd = np.ascontiguousarray(np.asarray(self.oa.io_to_dense, dtype=np.uint8)[np.frombuffer(query, dtype=np.uint8)])
        buf = qd if qd.size else np.zeros(1, np.uint8)
        occ = np.zeros(k + 1, dtype=np.uint64)
        cap = 1 << 16
        iv = np.zeros(3 * cap, dtype=np.uint64)
        steps = C.c_uint64()
        n = self.lib.emul_hamming(self.h, self.oa.num_searchable, self.n, buf.ctypes.data, len(query), k,
                                  occ.ctypes.data, iv.ctypes.data, cap, C.byref(steps))
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
