"""GPU tests of the Hamming search (gdx_count_many_hamming / gdx_cursors_many_hamming / gdx_locate_many_hamming) against a
naive scan of every window and the oracle, on every rank layout, storage type, construction route, with and without the
text section and the accelerators; its k = 0 form against the exact entry points; its errors; batches of several
chunks; concurrent calls; the C++ mirror.  On indexes of several rank superblocks (where a superblock's counts differ
from `count`), a homopolymer run, a repeat-rich genome slice and long queries: against the references of
tests/hamming_ref.py, and the node expansions (gdx_stats.lf_steps) against the host emulation of the same search, which
ties the device-only K32 expansion to the CPU-tested core.  Exact search on the same indexes against the oracle."""
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
from hamming_ref import (SUPERBLOCK, Cheapest, Naive, hamming_queries, hamming_texts, multi_superblock_texts,
                         window_queries)
from test_hamming_host import EmulIndex, build_emul

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
                          "-p", "no:cacheprovider", "-k",
                          "parity_with_naive_scan and (u32 or i32) or long_queries or errors or configurations or "
                          "boundary_lengths"],
                         env=env, capture_output=True, text=True, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]


# ---- indexes of several rank superblocks -----------------------------------------------------------------------

@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return build_emul(tmp_path_factory.mktemp("emul_hamming"))


# (rank_layout, rank_record_bytes): 0 = K32 (32-byte records of 64 positions), 1 = KG<B> (128 positions)
LAYOUTS = {
    "u8_until_0": (0, 32), "u8_until_2": (0, 32), "ascii_dna": (0, 32), "acg_n": (0, 32),
    "ascii_dna_with_n": (0, 32), "dna_n_searchable": (0, 32),
    "dna_rny": (1, 64),                     # KG<3>
    "dna_iupac_kept": (1, 96),              # KG<4>
    "protein20": (1, 128),                  # KG<5>
    "u8_until_40": (1, 192),                # KG<6>
    "ascii_printable": (1, 320),            # KG<7>
    "u8_ns4": (1, 640), "u8_until_254": (1, 640),  # KG<8>
}
LONG = (64, 65, 127, 128, 200, 255, 256)


def expect_layout(pidx, oidx, name):
    info = pidx.info()
    assert (info.rank_layout, info.rank_record_bytes) == LAYOUTS[name], name
    assert info.text_len == oidx.text_len
    return info


def check_with_steps(gdx, pidx, oidx, ref, ex, qs, k):
    """check_against_naive with another reference, and the node expansions of the locate call against the host
    emulation of the same search"""
    check_against_naive(gdx, pidx, oidx, ref, qs, k)
    assert pidx.stats().lf_steps == sum(ex.search(q, k)[2] for q in qs), k


def check_exact(pidx, oidx, oa, texts, seed):
    """exact search against the oracle, and extend_many on intervals that straddle each superblock boundary"""
    rng = random.Random(seed)
    util.assert_same_results(oidx, pidx, util.random_queries(rng, oa, texts, 300, 100, 40))
    syms = util.searchable_io_symbols(oa)
    n = oidx.text_len
    iv = []
    for b in range(SUPERBLOCK, n + 1, SUPERBLOCK):
        iv += [(b - 1, min(b + 1, n)), (b, min(b + 64, n)), (b - 128, b)]
        iv += [(b - rng.randrange(1, 5000), min(n, b + rng.randrange(1, 5000))) for _ in range(6)]
    sym = [rng.choice(syms) for _ in iv]
    s, e = pidx.extend_many_packed(np.array([a for a, _ in iv], dtype=np.uint64),
                                   np.array([b for _, b in iv], dtype=np.uint64), np.frombuffer(bytes(sym), np.uint8))
    assert list(zip(s.tolist(), e.tolist())) == [oidx.extend_query_front(x, c) for x, c in zip(iv, sym)]


def plan_for(ns):
    """[(k, query lengths, queries per length)] that keep the references cheap"""
    if ns == 1:  # a homopolymer: every window matches, one interval of the whole text per query
        return [(1, (10,), 1), (3, (40,), 1)]
    if ns <= 5:
        return [(1, (10, 24), 10), (2, (12, 30), 10), (3, (12, 16), 10), (3, LONG, 2)]
    if ns < 255:
        return [(1, (6, 12), 10), (2, (9,), 10), (3, (12,), 10), (3, LONG, 2)]
    return [(1, (3, 8), 10), (2, (9,), 6), (3, (12, 256), 2)]


SUPERBLOCK_CASES = [  # (alphabet, symbols)
    ("u8_until_0", 300_000), ("u8_until_2", 400_000), ("ascii_dna", 400_000), ("acg_n", 400_000),
    ("ascii_dna_with_n", 600_000), ("dna_n_searchable", 400_000), ("dna_rny", 400_000),
    ("dna_iupac_kept", 300_000), ("protein20", 400_000), ("u8_until_40", 300_000), ("ascii_printable", 300_000),
    ("u8_ns4", 300_000), ("u8_until_254", 400_000),
]


@pytest.mark.parametrize("name,total", SUPERBLOCK_CASES, ids=[c[0] for c in SUPERBLOCK_CASES])
def test_every_layout_on_several_superblocks(gdx, emul, name, total):
    oa = util.oracle_alphabet(name)
    seed = zlib.crc32(b"sb-" + name.encode())
    # (one searchable symbol: short texts, since a long homopolymer makes the oracle's suffix sort quadratic)
    texts = multi_superblock_texts(seed, oa, total, ntexts=6 if oa.num_searchable > 1 else 300)
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    pidx = build(gdx, texts, name, on_device=seed % 2 == 0)
    expect_layout(pidx, oidx, name)
    assert oidx.text_len > 4 * SUPERBLOCK
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    for k, lengths, nq in plan_for(oa.num_searchable):
        qs = [q for m in lengths for q in window_queries(seed + 31 * k + m, oa, texts, nq, m, k)]
        check_with_steps(gdx, pidx, oidx, ref, ex, qs, k)
    check_k0_equals_exact(pidx, window_queries(seed, oa, texts, 200 if oa.num_searchable > 1 else 4, 20, 0) + [b""])
    if LAYOUTS[name][0] == 0:  # the K32 expansion on borders of different superblocks, the derived child past 0
        _, derived = ex.layout()
        assert ex.cover[0] > 0, ex.cover
        assert (ex.cover[1] > 0) == (0 < derived <= oa.num_searchable), ex.cover
    check_exact(pidx, oidx, oa, texts, seed)


BOUNDARY_CASES = [(name, extra) for name in ("ascii_dna_with_n", "protein20") for extra in (-1, 0)]


@pytest.mark.parametrize("name,extra", BOUNDARY_CASES, ids=[f"{n}-n_plus_{1 + e}" for n, e in BOUNDARY_CASES])
def test_boundary_lengths(gdx, emul, name, extra):
    # text_len + 1 (extra = -1) or text_len (extra = 0) a multiple of the superblock: the last superblock filled up to
    # its end, and the record of position n alone in a superblock of its own
    oa = util.oracle_alphabet(name)
    seed = zlib.crc32(f"bl-{name}{extra}".encode())
    n = 4 * SUPERBLOCK + extra
    texts = multi_superblock_texts(seed, oa, n - 6)  # 6 texts, 6 sentinels
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    assert oidx.text_len == n and len(texts) == 6
    pidx = build(gdx, texts, name, on_device=extra == 0)
    expect_layout(pidx, oidx, name)
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    for k, lengths, nq in plan_for(oa.num_searchable)[:3]:
        qs = [q for m in lengths for q in window_queries(seed + k + m, oa, texts, nq, m, k)]
        check_with_steps(gdx, pidx, oidx, ref, ex, qs, k)
    check_exact(pidx, oidx, oa, texts, seed)


def test_interval_wider_than_u16(gdx, emul):
    # A x 70 000 across a superblock boundary: in-superblock u16 offsets near their maximum, and queries A x m whose
    # exact interval holds ~70 000 rows (the (end - start) << 2 packing and the fill of wide intervals in locate)
    oa = util.oracle_alphabet("ascii_dna_with_n")
    nrng = np.random.default_rng(70)
    rand = lambda n: nrng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), n, p=[.24] * 4 + [.04]).tobytes()  # noqa
    texts = [rand(40_000), rand(20_000) + b"A" * 70_000 + rand(50_000), b"", rand(30_000)]
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    pidx = build(gdx, texts, "ascii_dna_with_n")
    expect_layout(pidx, oidx, "ascii_dna_with_n")
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    qs = [b"A" * m for m in (1, 2, 12, 20, 100)] + [b"A" * 30 + b"C" + b"A" * 30, b"CA" + b"A" * 40]
    for k in range(4):
        check_with_steps(gdx, pidx, oidx, ref, ex, qs, k)
    assert ex.cover[2] > 0 and ex.cover[0] > 0, ex.cover
    cnt = pidx.count_many_hamming([b"A" * 20], 1)
    assert cnt[0, 0] > 65535


def test_repeat_rich_index(gdx, emul):
    # hg38-like repeat families at 6 Mbp: queries from repeat copies have hundreds of intervals (deep searches, large
    # pass-2 sort segments, many wide intervals); one batch of more than 2^20 queries, a sample of every chunk
    import torch
    if os.path.join(ROOT, "tools") not in sys.path:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
    import run_configs
    oa = util.oracle_alphabet("ascii_dna_with_n")
    text, _ = run_configs.make_repeat_rich_text(6_000_000, torch.device("cuda", 0))
    host = text.cpu().numpy()
    del text
    texts = [host[:2_500_000].tobytes(), b"", host[2_500_000:].tobytes()]
    oidx = O.OracleIndex.build(texts, oa, "u32", sampling_rate=4)
    pidx = build(gdx, texts, "ascii_dna_with_n", on_device=True)
    expect_layout(pidx, oidx, "ascii_dna_with_n")
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    rng = random.Random(77)
    # windows of repeat copies (at least 20 occurrences; 2 at m = 100, where copies diverge), 0..k substitutions
    most = 0
    for k, m in ((1, 20), (1, 100), (2, 20), (2, 40), (3, 20), (3, 40), (3, 100)):
        cand = [w.replace(b"N", b"A") for w in window_queries(rng.random(), oa, texts, 2000, m, 0)]
        c = oidx.count_many(cand, nthreads=0)
        reps = [w for w, x in zip(cand, c.tolist()) if x >= (20 if m < 100 else 2)][:6]
        assert len(reps) >= 3, (k, m)
        qs = []
        for w in reps:
            w = bytearray(w)
            for _ in range(rng.randrange(k + 1)):
                w[rng.randrange(m)] = rng.choice(b"ACGT")
            qs.append(bytes(w))
        check_with_steps(gdx, pidx, oidx, ref, ex, qs, k)
        data, off = O.pack(qs)
        ioff = pidx.cursors_many_hamming_packed(data, off, k)[0]
        most = max(most, int(np.diff(ioff).max()))
    assert most >= 100, most
    # more than 2^20 queries at k = 1: a sample of each chunk and the first and last query against the reference
    nrng = np.random.default_rng(78)
    nq, m = CHUNK + 40_000, 30
    arr = np.frombuffer(b"".join(texts), dtype=np.uint8)
    starts = nrng.integers(0, arr.size - m, nq)
    qmat = arr[starts[:, None] + np.arange(m)].copy()
    qmat[qmat == ord("N")] = ord("C")
    flip = np.flatnonzero(nrng.random(nq) < 0.5)
    qmat[flip, nrng.integers(0, m, flip.size)] = ord("G")
    data = np.ascontiguousarray(qmat.reshape(-1))
    off = np.arange(nq + 1, dtype=np.uint64) * m
    counts = pidx.count_many_hamming_packed(data, off, 1)
    ioff, s, e, d = pidx.cursors_many_hamming_packed(data, off, 1)
    hoff, hits = pidx.locate_many_hamming_packed(data, off, 1)
    assert np.array_equal(np.diff(hoff), counts.sum(axis=1))
    sample = sorted(set(rng.sample(range(CHUNK), 40) + rng.sample(range(CHUNK, nq), 40) + [0, CHUNK - 1, CHUNK, nq - 1]))
    for i in sample:
        occ, ivs, _ = ref.expected(bytes(qmat[i]), 1)
        assert counts[i].tolist() == occ, i
        a, b = int(ioff[i]), int(ioff[i + 1])
        assert list(zip(s[a:b].tolist(), e[a:b].tolist(), d[a:b].tolist())) == ivs, i
        a, b = int(hoff[i]), int(hoff[i + 1])
        assert [tuple(h) for h in hits[a:b].tolist()] == [h for x, y, _ in ivs for h in oidx.locate_interval(x, y)], i
    # the sampled queries alone: node expansions against the host emulation
    check_with_steps(gdx, pidx, oidx, ref, ex, [bytes(qmat[i]) for i in sample], 1)


CONFIGS = [  # (alphabet, storage, on_device, sampling rate, dense suffix array, text section)
    ("ascii_dna_with_n", "u32", False, 1, True, True),
    ("ascii_dna_with_n", "i64", True, 3, False, True),
    ("ascii_dna_with_n", "u32", True, 32, False, False),
    ("ascii_dna_with_n", "i64", False, 4, True, False),
    ("protein20", "u32", True, 1, False, False),
    ("protein20", "i64", False, 3, True, True),
    ("protein20", "u32", False, 32, True, False),
    ("protein20", "i64", True, 4, False, True),
]


@pytest.mark.parametrize("name,storage,on_device,rate,dense,text", CONFIGS,
                         ids=["-".join(str(x) for x in c) for c in CONFIGS])
def test_configurations_on_several_superblocks(gdx, emul, name, storage, on_device, rate, dense, text):
    oa = util.oracle_alphabet(name)
    seed = zlib.crc32("-".join(str(x) for x in (name, storage, on_device, rate, dense, text)).encode())
    texts = multi_superblock_texts(seed, oa, 300_000)
    oidx = O.OracleIndex.build(texts, oa, storage, sampling_rate=rate)
    cfg = (gdx.FmIndexConfig(storage).suffix_array_sampling_rate(rate).construct_on_device(on_device, verify=on_device)
           .keep_text(text).dense_suffix_array(dense))
    pidx = cfg.construct_index(texts, util.product_alphabet(gdx, name))
    if dense:
        pidx.set_dense_suffix_array(True)
    info = expect_layout(pidx, oidx, name)
    assert info.sampling_rate == rate
    assert (info.dense_suffix_array_bytes > 0) == dense and (info.text_bytes > 0) == text
    ref, ex = Cheapest(oidx, oa), EmulIndex(emul, oidx, oa)
    for k, lengths, nq in plan_for(oa.num_searchable):
        qs = [q for m in lengths for q in window_queries(seed + 7 * k + m, oa, texts, min(nq, 4), m, k)]
        check_with_steps(gdx, pidx, oidx, ref, ex, qs, k)
    check_exact(pidx, oidx, oa, texts, seed)
