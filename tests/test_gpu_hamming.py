"""GPU tests of the Hamming search (gdx_count_many_hamming / gdx_cursors_many_hamming / gdx_locate_many_hamming) against a
naive scan of every window and the oracle, on every rank layout, storage type, construction route, with and without the
text section and the accelerators; its k = 0 form against the exact entry points; its errors; batches of several
chunks; concurrent calls; the C++ mirror."""
import ctypes as C
import os
import random
import subprocess
import sys
import threading
import zlib

import numpy as np
import pytest

from oracle import oracle as O
import gdx_testutil as util
from hamming_ref import Naive, hamming_queries, hamming_texts

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 1 << 20  # kHammingChunkQueries in api.cu


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    return genedex_b200


def build(gdx, texts, name, storage="u32", on_device=False, depth=0, variant="default"):
    cfg = gdx.FmIndexConfig(storage).suffix_array_sampling_rate(4).lookup_table_depth(depth)
    cfg = cfg.construct_on_device(on_device, verify=on_device)
    if variant == "no_text":
        cfg = cfg.keep_text(False)
    if variant == "accel_off":
        cfg = cfg.dense_suffix_array(False).seed_table(False).row_context_table(False)
    pidx = cfg.construct_index(texts, util.product_alphabet(gdx, name))
    if variant == "accel_on":
        pidx.set_dense_suffix_array(True)
        pidx.set_seed_table_depth(depth + 3)
        try:
            pidx.set_row_context_table(True)
        except gdx.GenedexError:
            pass  # needs at most 4 searchable symbols
    if variant == "lf_only":
        pidx.set_text_verification(False)
    return pidx


def check_against_naive(gdx, pidx, oidx, naive, qs, k):
    data, off = O.pack(qs)
    counts = pidx.count_many_hamming_packed(data, off, k)
    ioff, starts, ends, mism = pidx.cursors_many_hamming_packed(data, off, k)
    hoff, hits = pidx.locate_many_hamming_packed(data, off, k)
    assert counts.shape == (len(qs), k + 1)
    for i, q in enumerate(qs):
        occ, ivs, _ = naive.expected(q, k)
        assert counts[i].tolist() == occ, (q, k)
        a, b = int(ioff[i]), int(ioff[i + 1])
        got = list(zip(starts[a:b].tolist(), ends[a:b].tolist(), mism[a:b].tolist()))
        assert got == ivs, (q, k)
        want_hits = [h for s, e, _ in ivs for h in oidx.locate_interval(s, e)]
        a, b = int(hoff[i]), int(hoff[i + 1])
        assert [tuple(h) for h in hits[a:b].tolist()] == want_hits, (q, k)
    assert int(hoff[-1]) == hits.shape[0] and int(ioff[-1]) == starts.size


def check_k0_equals_exact(pidx, qs):
    data, off = O.pack(qs)
    s, e = pidx.cursors_many_packed(data, off)
    c = pidx.count_many_packed(data, off)
    loff, lhits = pidx.locate_many_packed(data, off)
    hc = pidx.count_many_hamming_packed(data, off, 0)
    ioff, hs, he, hm = pidx.cursors_many_hamming_packed(data, off, 0)
    hoff, hhits = pidx.locate_many_hamming_packed(data, off, 0)
    assert np.array_equal(hc[:, 0], c)
    nonempty = e > s
    assert np.array_equal(np.diff(ioff), nonempty.astype(np.uint64))
    assert np.array_equal(hs, s[nonempty]) and np.array_equal(he, e[nonempty]) and not hm.any()
    assert np.array_equal(hoff, loff) and np.array_equal(hhits, lhits)


CASES = [
    # (alphabet, storage, on_device, lookup depth, variant)
    ("ascii_dna_with_n", "u32", False, 0, "default"),
    ("ascii_dna_with_n", "i32", True, 3, "no_text"),
    ("ascii_dna_with_n", "i64", False, 2, "accel_on"),
    ("dna_n_searchable", "u32", True, 0, "default"),       # K32, derived rank of a searchable symbol
    ("dna_n_searchable", "i64", False, 3, "accel_off"),
    ("acg_n", "i32", False, 2, "lf_only"),                  # K32, 3 searchable symbols
    ("dna_rny", "u32", True, 4, "accel_on"),                # KG<3>
    ("dna_iupac_kept", "i32", False, 0, "no_text"),          # KG<4>
    ("dna_iupac_gaps", "i64", True, 2, "default"),          # KG<5>, 8-bit text
    ("u8_ns4", "u32", False, 3, "accel_off"),               # KG<8>
    ("protein20", "u32", True, 2, "accel_on"),              # KG<5>, 20 searchable symbols
    ("protein20", "i64", False, 0, "lf_only"),
]


@pytest.mark.parametrize("name,storage,on_device,depth,variant", CASES,
                         ids=["-".join(str(x) for x in c) for c in CASES])
def test_parity_with_naive_scan(gdx, name, storage, on_device, depth, variant):
    oa = util.oracle_alphabet(name)
    rng = random.Random(zlib.crc32(f"{name}-{storage}-{depth}-{variant}".encode()))
    texts = hamming_texts(rng, oa, 4, 1500)
    oidx = O.OracleIndex.build(texts, oa, storage, sampling_rate=4)
    pidx = build(gdx, texts, name, storage, on_device, depth, variant)
    naive = Naive(oidx, texts, oa)
    for k in range(4):
        max_len = 7 if oa.num_searchable > 5 and k >= 2 else 12
        check_against_naive(gdx, pidx, oidx, naive, hamming_queries(rng, oa, texts, 60, max_len, k), k)
    # k = 0 against the exact entry points, queries of searchable symbols of every length up to the limit
    qs = hamming_queries(rng, oa, texts, 400, 40, 2) + [b""]
    check_k0_equals_exact(pidx, qs)


def test_long_queries_and_k_at_least_m(gdx):
    oa = util.oracle_alphabet("ascii_dna_with_n")
    rng = random.Random(3)
    texts = hamming_texts(rng, oa, 3, 3000, p_other=0.02)
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    pidx = build(gdx, texts, "ascii_dna_with_n")
    naive = Naive(oidx, texts, oa)
    t = max(texts, key=len)
    long_qs = []
    for m in (64, 100, 255, 256):
        if len(t) >= m:
            p = rng.randrange(len(t) - m + 1)
            w = bytearray(t[p:p + m].replace(b"N", b"A"))
            w[rng.randrange(m)] = ord("C")
            long_qs.append(bytes(w))
    check_against_naive(gdx, pidx, oidx, naive, long_qs + [b"A", b"AC", b"ACG", b""], 3)


def expect_error(gdx, fn, status, query=None):
    with pytest.raises(gdx.GenedexError) as ei:
        fn()
    assert ei.value.status == status, str(ei.value)
    if query is not None:
        assert int(gdx._lib.load().gdx_last_error_query()) == query, str(ei.value)


def all_forms(pidx, data, off, k, fixed_len=0, nq=None):
    return [lambda: pidx.count_many_hamming_packed(data, off, k, fixed_len, nq),
            lambda: pidx.cursors_many_hamming_packed(data, off, k, fixed_len, nq),
            lambda: pidx.locate_many_hamming_packed(data, off, k, fixed_len, nq)]


def test_errors(gdx):
    L = gdx._lib
    texts = [b"ACGTNACGTACGGT" * 50, b"GATTACA" * 30]
    pidx = build(gdx, texts, "ascii_dna_with_n")
    ok = [b"ACGT", b"acgt", b"GATTACA"]
    for bad, st in [(b"ACNT", L.GDX_ERR_INVALID_SYMBOL), (b"ACXT", L.GDX_ERR_INVALID_SYMBOL),
                    (b"A" * 257, L.GDX_ERR_UNSUPPORTED)]:
        qs = ok + [bad] + ok + [b"NNN"]
        data, off = O.pack(qs)
        for fn in all_forms(pidx, data, off, 1):
            expect_error(gdx, fn, st, 3)
    data, off = O.pack(ok)
    for fn in all_forms(pidx, data, off, 4):
        expect_error(gdx, fn, L.GDX_ERR_BAD_ARG)
    # broken offsets (decreasing, or leaving the batch)
    for broken in ([0, 4, 2, 8], [0, 4, 9, 8]):
        boff = np.array(broken, dtype=np.uint64)
        bdata = np.frombuffer(b"ACGTACGTACGT", dtype=np.uint8).copy()
        for fn in all_forms(pidx, bdata, boff, 1):
            expect_error(gdx, fn, L.GDX_ERR_BAD_ARG, 1)
    # fixed-length batches longer than the limit
    fdata = np.frombuffer(b"A" * 600, dtype=np.uint8).copy()
    for fn in all_forms(pidx, fdata, None, 1, fixed_len=300, nq=2):
        expect_error(gdx, fn, L.GDX_ERR_UNSUPPORTED, 0)
    # 2-bit packed input is not taken
    q = L.gdx_queries(data.ctypes.data, off.ctypes.data, 0, len(ok), L.GDX_QUERIES_PACKED_2BIT, 0)
    out = np.zeros(len(ok) * 2, dtype=np.uint64)
    assert pidx._lib.gdx_count_many_hamming(pidx.handle, C.byref(q), 1, out.ctypes.data) == L.GDX_ERR_UNSUPPORTED
    # a valid batch still works on the same handle
    assert pidx.count_many_hamming(ok, 1).shape == (3, 2)


def test_error_names_smallest_query_in_a_later_chunk(gdx):
    L = gdx._lib
    texts = [bytes(random.Random(5).choice(b"ACGT") for _ in range(20000))]
    pidx = build(gdx, texts, "ascii_dna_with_n")
    n = 2 * CHUNK + 1000
    base = [b"ACGTACGTAC"] * n

    def run(edits, k, want_status, want_query):
        qs = list(base)
        for i, q in edits.items():
            qs[i] = q
        data, off = O.pack(qs)
        for fn in all_forms(pidx, data, off, k):
            expect_error(gdx, fn, want_status, want_query)

    # invalid symbol in the second chunk before a long query in the third
    run({CHUNK + 5: b"ACGNA", 2 * CHUNK + 7: b"A" * 300, 2 * CHUNK + 9: b"X"}, 1, L.GDX_ERR_INVALID_SYMBOL, CHUNK + 5)
    # a long query in front of the invalid symbol
    run({CHUNK + 3: b"C" * 257, CHUNK + 5: b"ACGNA"}, 2, L.GDX_ERR_UNSUPPORTED, CHUNK + 3)


def test_batch_of_several_chunks(gdx):
    oa = util.oracle_alphabet("ascii_dna_with_n")
    rng = random.Random(9)
    nrng = np.random.default_rng(9)
    text = nrng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 60000)
    text[1000:1100] = ord("N")
    texts = [text.tobytes()]
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    pidx = build(gdx, texts, "ascii_dna_with_n")
    naive = Naive(oidx, texts, oa)
    n, m = 2 * CHUNK + 12345, 12
    starts = nrng.integers(0, text.size - m, n)
    qmat = text[starts[:, None] + np.arange(m)].copy()
    qmat[qmat == ord("N")] = ord("G")
    flip = nrng.random(n) < 0.5  # one substitution in half of them
    qmat[np.flatnonzero(flip), nrng.integers(0, m, flip.sum())] = ord("T")
    data = np.ascontiguousarray(qmat.reshape(-1))
    # k = 0 equals the exact path on the whole batch (fixed-length form)
    c = pidx.count_many_packed(data, None, m, n)
    hc = pidx.count_many_hamming_packed(data, None, 0, m, n)
    assert np.array_equal(hc[:, 0], c)
    # k = 1 on the whole batch, a sample of every chunk against the naive scan
    off = np.arange(n + 1, dtype=np.uint64) * m
    counts = pidx.count_many_hamming_packed(data, off, 1)
    ioff, s, e, d = pidx.cursors_many_hamming_packed(data, off, 1)
    hoff, hits = pidx.locate_many_hamming_packed(data, off, 1)
    assert np.array_equal(np.diff(hoff), counts.sum(axis=1))
    sample = sorted(set(rng.sample(range(CHUNK), 100) + rng.sample(range(CHUNK, 2 * CHUNK), 100) +
                        rng.sample(range(2 * CHUNK, n), 100) + [CHUNK - 1, CHUNK, 2 * CHUNK, n - 1]))
    for i in sample:
        q = bytes(qmat[i])
        occ, ivs, _ = naive.expected(q, 1)
        assert counts[i].tolist() == occ
        a, b = int(ioff[i]), int(ioff[i + 1])
        assert list(zip(s[a:b].tolist(), e[a:b].tolist(), d[a:b].tolist())) == ivs
        a, b = int(hoff[i]), int(hoff[i + 1])
        assert [tuple(h) for h in hits[a:b].tolist()] == [h for x, y, _ in ivs for h in oidx.locate_interval(x, y)]
    st = pidx.stats()
    assert st.queries == n and st.hits == hits.shape[0] and st.lf_steps >= n


def test_concurrent_calls_on_one_handle(gdx):
    oa = util.oracle_alphabet("ascii_dna_with_n")
    rng = random.Random(21)
    texts = hamming_texts(rng, oa, 3, 20000, p_other=0.01)
    pidx = build(gdx, texts, "ascii_dna_with_n")
    qs = hamming_queries(rng, oa, texts, 20000, 30, 2)
    data, off = O.pack(qs)
    want = (pidx.count_many_hamming_packed(data, off, 2), pidx.locate_many_hamming_packed(data, off, 2),
            pidx.count_many_packed(data, off), pidx.locate_many_packed(data, off))
    errors = []

    def worker(t):
        try:
            for r in range(4):
                if (t + r) % 2:
                    assert np.array_equal(pidx.count_many_hamming_packed(data, off, 2), want[0])
                    h = pidx.locate_many_hamming_packed(data, off, 2)
                    assert np.array_equal(h[0], want[1][0]) and np.array_equal(h[1], want[1][1])
                else:
                    assert np.array_equal(pidx.count_many_packed(data, off), want[2])
                    h = pidx.locate_many_packed(data, off)
                    assert np.array_equal(h[0], want[3][0]) and np.array_equal(h[1], want[3][1])
        except Exception as ex:  # noqa: BLE001 -- reported by the main thread
            errors.append(ex)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(6)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors


CPP = r'''
#include <cstdio>
#include <string>
#include <vector>
#include "genedex_b200.hpp"
int main() {
    std::vector<std::string> texts{"ACGTACGTTTACGAACGT", "GGACGTA"};
    gdx::FmIndex index = gdx::FmIndexConfig<gdx::U32>().construct_index(texts, gdx::alphabet::ascii_dna_with_n());
    std::vector<std::string> qs{"ACGT", "ACGA", "acg", ""};
    auto counts = index.count_many_hamming(qs, 1);
    auto cursors = index.cursors_many_hamming(qs, 1);
    auto hits = index.locate_many_hamming(qs, 1);
    for (size_t i = 0; i < qs.size(); ++i) {
        std::printf("q%zu counts", i);
        for (size_t c : counts[i]) std::printf(" %zu", c);
        std::printf(" intervals");
        for (auto &cm : cursors[i]) std::printf(" %llu:%llu:%u", (unsigned long long)cm.first.interval().first,
                                                (unsigned long long)cm.first.interval().second, cm.second);
        std::printf(" hits");
        for (auto &h : hits[i]) std::printf(" %zu:%zu", h.text_id, h.position);
        std::printf("\n");
    }
    return 0;
}
'''


def test_cpp_mirror(gdx, tmp_path):
    src = tmp_path / "hamming.cpp"
    src.write_text(CPP)
    exe = tmp_path / "hamming"
    libdir = os.path.join(ROOT, "genedex_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), str(src),
                           "-L", libdir, "-lgenedex_b200", f"-Wl,-rpath,{libdir}", "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    texts = [b"ACGTACGTTTACGAACGT", b"GGACGTA"]
    pidx = gdx.FmIndexConfig("u32").construct_index(texts, gdx.alphabet.ascii_dna_with_n())
    qs = [b"ACGT", b"ACGA", b"acg", b""]
    counts = pidx.count_many_hamming(qs, 1)
    cursors = pidx.cursors_many_hamming(qs, 1)
    hits = pidx.locate_many_hamming(qs, 1)
    want = []
    for i in range(len(qs)):
        want.append(f"q{i} counts " + " ".join(str(int(c)) for c in counts[i]) + " intervals" +
                    "".join(f" {c.interval[0]}:{c.interval[1]}:{d}" for c, d in cursors[i]) + " hits" +
                    "".join(f" {h.text_id}:{h.position}" for h in hits[i]))
    assert out == want
    assert sum(int(c[1]) for c in counts) > 0


@pytest.mark.skipif(os.environ.get("GDX_FORCE_WIDE") == "1", reason="already the wide run")
def test_wide_path():
    # the 64-bit sample / lookup paths, on a subset of this file in a process of its own
    env = dict(os.environ, GDX_FORCE_WIDE="1")
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x",
                          "-p", "no:cacheprovider", "-k", "parity_with_naive_scan and (u32 or i32) or long_queries or errors"],
                         env=env, capture_output=True, text=True, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
