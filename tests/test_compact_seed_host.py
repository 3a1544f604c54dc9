"""CPU tests of the compact seed level (genedex_b200/csrc/compact_seed.h) and of its policy (accel_policy.h), built on
the host with g++: the SA-order index from packed codes, the group decode with and without exception records, and a
table built from a brute-force suffix sort, checked against S(i) and width(i) counted directly from the text.
No GPU is used here."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U64P = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")
U32P = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
U8P = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
SLOTS = 224


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("emul_compact_seed") / "libcompactseed.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Wno-unknown-pragmas", "-shared", "-fPIC", "-o",
                           str(out), os.path.join(ROOT, "tests", "host_emul", "compact_seed_emul.cpp")])
    lib = C.CDLL(str(out))
    lib.emul_cs_index_from_codes.restype = C.c_uint64
    lib.emul_cs_index_from_codes.argtypes = [C.c_uint64, C.c_uint32]
    lib.emul_cs_decode.restype = None
    lib.emul_cs_decode.argtypes = [U64P, C.c_uint32, U32P, U64P]
    lib.emul_cs_build.restype = C.c_int64
    lib.emul_cs_build.argtypes = [U8P, C.c_uint64, U32P, C.c_uint32, C.c_uint32, U8P, U32P]
    lib.emul_cs_policy.restype = None
    lib.emul_cs_policy.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                   C.c_uint64, C.c_uint64, C.c_uint64, U64P]
    return lib


def test_index_from_packed_codes(lib):
    rng = random.Random(1)
    for _ in range(3000):
        d = rng.randrange(1, 33)
        codes = [rng.randrange(4) for _ in range(d)]
        v = sum(c << (2 * j) for j, c in enumerate(codes))
        want = 0
        for c in codes:  # x_0 most significant
            want = want * 4 + c
        assert lib.emul_cs_index_from_codes(v, d) == want


def make_group(rng, with_record):
    """(words, pool, widths, gaps) of a random group: base + fields, and a record when some slot needs one"""
    widths = [rng.choice([0, 0, 1, 1, 1, 2] + ([3, 7, 70_000] if with_record else [])) for _ in range(SLOTS)]
    gaps = [rng.choice([0] * 12 + [1, 5]) if with_record else 0 for _ in range(SLOTS)]
    base = rng.randrange(1 << 31)
    fields = 0
    for j, w in enumerate(widths):
        fields |= min(w, 3) << (2 * j)
    exc = [(j, widths[j], gaps[j]) for j in range(SLOTS) if widths[j] >= 3 or gaps[j] > 0]
    pool = [rng.randrange(1 << 32) for _ in range(rng.randrange(5))]  # records of other groups in front
    off = 0xFFFFFFFF
    if exc:
        off = len(pool)
        pool.append(len(exc))
        for t in exc:
            pool.extend(t)
    words = np.zeros(8, dtype=np.uint64)
    words[0] = base | (off << 32)
    for k in range(7):
        words[1 + k] = (fields >> (64 * k)) & (2 ** 64 - 1)
    return words, np.array(pool + [0], dtype=np.uint32), base, widths, gaps


@pytest.mark.parametrize("with_record", [False, True])
def test_group_decode(lib, with_record):
    rng = random.Random(2 + with_record)
    out = np.zeros(2, dtype=np.uint64)
    for _ in range(40):
        words, pool, base, widths, gaps = make_group(rng, with_record)
        start = base
        for j in range(SLOTS):
            lib.emul_cs_decode(words, j, pool, out)
            assert (int(out[0]), int(out[1])) == (start, start + widths[j]), j
            start += widths[j] + gaps[j]


DENSE = {ord("A"): 1, ord("C"): 2, ord("G"): 3, ord("T"): 4, ord("N"): 5}
NS = 4


def concat(texts):
    """dense symbols of the texts, each followed by its sentinel (0)"""
    return np.array([s for t in texts for s in [DENSE[b] for b in t] + [0]], dtype=np.uint8)


def suffix_array(text, d, brute):
    n = text.size
    raw = text.tobytes()
    if brute:  # full suffixes
        return np.array(sorted(range(n), key=lambda i: raw[i:]), dtype=np.uint32)
    # the first d symbols decide everything the level holds (long single-symbol texts)
    return np.array(sorted(range(n), key=lambda i: raw[i:i + d] + b"\0" * max(0, i + d - n)), dtype=np.uint32)


def direct_intervals(text, d):
    """S(i) and width(i) of every d-mer, from the definition: rows whose d-prefix (sentinel = 0, 0 past the end)
    sorts before K_i, and rows whose d-prefix is K_i"""
    n = text.size
    pad = np.concatenate([text, np.zeros(d, dtype=np.uint8)]).astype(np.int64)
    # d-prefix as a base-6 number keeps its order (symbols 0..5)
    key = np.zeros(n, dtype=np.int64)
    for j in range(d):
        key = key * 6 + pad[j:j + n]
    key.sort()
    kmers = np.arange(NS ** d, dtype=np.int64)
    k6 = np.zeros_like(kmers)
    for j in range(d):
        k6 = k6 * 6 + ((kmers // NS ** (d - 1 - j)) % NS + 1)
    S = np.searchsorted(key, k6, side="left")
    W = np.searchsorted(key, k6, side="right") - S
    return S, W


def build_table(lib, text, sa, d):
    groups_n = (NS ** d + SLOTS - 1) // SLOTS
    groups = np.zeros(groups_n * 64, dtype=np.uint8)
    pool = np.zeros(4 * text.size + 4, dtype=np.uint32)
    used = lib.emul_cs_build(text, text.size, sa, d, NS, groups, pool)
    assert used >= 0, "rows out of order"
    return groups.view(np.uint64).reshape(groups_n, 8), pool, used


TEXTS = {
    "n_runs": lambda rng: [bytes(rng.choice(b"ACGT") for _ in range(900)) + b"N" * 7 + bytes(rng.choice(b"ACGT") for _ in range(300))
                           + b"NN" + b"ACG" + b"N" * 30 + bytes(rng.choice(b"ACGT") for _ in range(200))],
    "several_texts": lambda rng: [bytes(rng.choice(b"ACGTN") for _ in range(rng.randrange(1, 400))) for _ in range(6)],
    "repeats": lambda rng: [(b"ACGTTGCA" * 60) + bytes(rng.choice(b"ACGT") for _ in range(100)), b"GATTACA" * 40],
    "shorter_than_d": lambda rng: [b"AC", b"T", b"GGA", b"N", b""],
}


@pytest.mark.parametrize("name", sorted(TEXTS))
@pytest.mark.parametrize("d", [3, 5, 6])
def test_built_table_gives_every_interval(lib, name, d):
    rng = random.Random(len(name) * 7 + d)
    text = concat(TEXTS[name](rng))
    sa = suffix_array(text, d, brute=True)
    words, pool, used = build_table(lib, text, sa, d)
    S, W = direct_intervals(text, d)
    out = np.zeros(2, dtype=np.uint64)
    for k in range(NS ** d):
        lib.emul_cs_decode(np.ascontiguousarray(words[k // SLOTS]), k % SLOTS, pool, out)
        assert (int(out[0]), int(out[1])) == (S[k], S[k] + W[k]), k
    if name in ("n_runs", "repeats"):
        assert used > 0  # widths >= 3 or gaps: exception records


def test_a_dmer_of_more_than_65536_rows(lib):
    d = 6
    text = concat([b"A" * 70_000, b"ACGTN" * 10, b"C" * 100])
    sa = suffix_array(text, d, brute=False)
    words, pool, used = build_table(lib, text, sa, d)
    assert used > 0
    S, W = direct_intervals(text, d)
    assert W.max() > 1 << 16
    out = np.zeros(2, dtype=np.uint64)
    for k in range(NS ** d):
        lib.emul_cs_decode(np.ascontiguousarray(words[k // SLOTS]), k % SLOTS, pool, out)
        assert (int(out[0]), int(out[1])) == (S[k], S[k] + W[k]), k


def seed_entries(ns, d):
    e = 1
    for _ in range(d):
        e *= ns
        if e > 1 << 36:
            return 0
    return e


def test_policy(lib):
    rng = random.Random(4)
    out = np.zeros(3, dtype=np.uint64)
    for _ in range(20_000):
        n = rng.choice([0, 1, rng.randrange(2, 1000), rng.randrange(1000, 1 << 32), rng.randrange(1 << 32, 1 << 34)])
        ns = rng.choice([1, 2, 3, 4, 5, 20])
        wide, text = rng.random() < 0.2, rng.random() < 0.8
        seed = rng.choice([0, rng.randrange(1, 20)])
        budget = rng.choice([0, rng.randrange(1 << 36)])
        used, free = rng.randrange(1 << 35), rng.choice([2 ** 64 - 1, rng.randrange(1 << 38)])
        d, rec = rng.randrange(1, 40), rng.randrange(1 << 30)
        lib.emul_cs_policy(n, budget, ns, int(wide), int(text), seed, d, rec, used, free, out)
        possible = seed > 0 and not wide and 0 < n < 1 << 32 and text and ns >= 2
        depth = 0
        if possible:
            depth = seed
            while seed_entries(ns, depth + 1) and seed_entries(ns, depth + 1) <= 32 * n:
                depth += 1
            depth = depth if depth > seed else 0
        room = max(budget - used, 0) if budget else (0 if free == 2 ** 64 - 1 else 2 * (free // 4))
        fits = (seed_entries(ns, d) + SLOTS - 1) // SLOTS * 64 + rec <= room
        assert (bool(out[0]), int(out[1]), bool(out[2])) == (possible, depth, fits)
    # the headline DNA index: seed depth 16, compact level 18; an index at 2 % of it: seed depth 13, compact level 15
    lib.emul_cs_policy(3_100_000_000, 0, 4, 0, 1, 16, 18, 0, 0, 1 << 40, out)
    assert int(out[1]) == 18
    lib.emul_cs_policy(62_000_000, 0, 4, 0, 1, 13, 15, 0, 0, 1 << 40, out)
    assert int(out[1]) == 15
