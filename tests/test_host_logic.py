"""CPU tests of the host-side logic of the product: the C ABI loads and exports every declared
symbol, host construction (SA-IS) equals the oracle's suffix array, and the device rank-record
arithmetic (rank_core.h, emulated on the host) equals the oracle's rank for every symbol/position.
No GPU compute is called here."""
import ctypes as C
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETTINGS = dict(deadline=None, suppress_health_check=list(HealthCheck))


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    return genedex_b200


def test_library_exports_every_declared_symbol(gdx):
    header = open(os.path.join(ROOT, "include", "genedex_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)  # drop comments
    declared = set(re.findall(r"\b(gdx_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    lib = C.CDLL(gdx._lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared in the header but not exported"
    assert declared == set(gdx._lib.PROTOTYPES), "Python prototypes and header disagree"
    assert lib.gdx_abi_version() == gdx._lib.GDX_ABI_VERSION == 2
    assert lib.gdx_index_header_bytes() > 256


def test_struct_sizes_match_the_header(gdx, tmp_path):
    # compile a tiny C program against the header and compare sizeof() with the ctypes mirrors
    src = tmp_path / "sizes.c"
    src.write_text('#include <stdio.h>\n#include "genedex_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(gdx_alphabet),sizeof(gdx_config),sizeof(gdx_hit),sizeof(gdx_queries),sizeof(gdx_parts),'
                   'sizeof(gdx_index_info),sizeof(gdx_stats));return 0;}\n')
    exe = tmp_path / "sizes"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    L = gdx._lib
    want = [C.sizeof(t) for t in (L.gdx_alphabet, L.gdx_config, L.gdx_hit, L.gdx_queries, L.gdx_parts,
                                  L.gdx_index_info, L.gdx_stats)]
    assert got == want


def test_no_cpu_fallback():
    # in a process that sees no CUDA device (CUDA_VISIBLE_DEVICES=""), so the check also runs where a GPU is present
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import genedex_b200 as gdx\n"
            "try:\n"
            "    gdx.FmIndexConfig('i32').construct_index([b'ACGT'], gdx.alphabet.ascii_dna())\n"
            "except gdx.GenedexError as e:\n"
            "    print(e)\n"
            "else:\n"
            "    sys.exit('an index was built without a CUDA device')\n" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "no CPU fallback" in out.stdout


def _host_sa(gdx, dense, sigma):
    lib = gdx._lib.load()
    t = np.ascontiguousarray(dense, dtype=np.uint8)
    out = np.zeros(max(t.size, 1), dtype=np.uint64)
    rc = lib.gdx_suffix_array(t.ctypes.data, t.size, sigma, gdx._lib.GDX_CONSTRUCT_HOST, -1, out.ctypes.data)
    assert rc == 0
    return out[:t.size].tolist()


@settings(max_examples=150, **SETTINGS)
@given(data=st.data())
def test_host_sais_equals_naive_and_oracle(gdx, data):
    kind = data.draw(st.sampled_from(["random", "runs", "periodic", "wide"]))
    if kind == "random":
        sigma = 6
        dense = data.draw(st.lists(st.integers(0, 5), min_size=1, max_size=400))
    elif kind == "runs":
        sigma = 6
        parts = data.draw(st.lists(st.tuples(st.integers(0, 5), st.integers(1, 90)), min_size=1, max_size=10))
        dense = [c for c, k in parts for _ in range(k)]
    elif kind == "periodic":
        sigma = 4
        unit = data.draw(st.lists(st.integers(1, 3), min_size=1, max_size=5))
        dense = unit * data.draw(st.integers(1, 80)) + [0]
    else:
        sigma = 256
        dense = data.draw(st.lists(st.integers(0, 255), min_size=1, max_size=300))
    assert _host_sa(gdx, dense, sigma) == O.naive_suffix_array(dense)


def test_host_sais_medium_equals_oracle(gdx):
    rng = np.random.default_rng(5)
    text = rng.integers(1, 5, 200_000, dtype=np.uint8)
    text[1000:9000] = 5           # a long run of N
    text[50_000] = 0
    text[50_001] = 0              # an empty text in the middle
    text[-1] = 0
    io = np.frombuffer(b"\x00ACGTN", dtype=np.uint8)[text]
    # split at sentinels to rebuild the same dense text through the oracle
    texts = bytes(io.tobytes()).split(b"\x00")[:-1]
    idx = O.OracleIndex.build(texts, O.ALPHABETS["ascii_dna_with_n"](), "u32", sampling_rate=1)
    assert np.array_equal(idx.dense_text(), text)
    assert _host_sa(gdx, text, 6) == idx.suffix_array().tolist()


# ---- device record arithmetic, emulated on the host ---------------------------------------------------
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    out = tmp_path_factory.mktemp("emul") / "libemul.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(ROOT, "tests", "host_emul", "emul.cpp")])
    lib = C.CDLL(str(out))
    lib.emul_build.restype = C.c_void_p
    lib.emul_build.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.emul_free.argtypes = [C.c_void_p]
    lib.emul_lf.restype = C.c_uint64
    lib.emul_lf.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64]
    lib.emul_symbol_at.restype = C.c_uint32
    lib.emul_symbol_at.argtypes = [C.c_void_p, C.c_uint64]
    lib.emul_layout.argtypes = [C.c_void_p, C.c_void_p]
    return lib


def _check_records(emul, bwt, sigma, positions=None):
    bwt = np.ascontiguousarray(bwt, dtype=np.uint8)
    n = bwt.size
    keep = bwt if n else np.zeros(1, np.uint8)
    freq = np.bincount(bwt, minlength=sigma + 1).astype(np.uint64)
    count = np.zeros(sigma + 1, dtype=np.uint64)
    count[1:] = np.cumsum(freq[:sigma])
    border_rows = np.flatnonzero(bwt == 0).astype(np.uint64)
    br = border_rows if border_rows.size else np.zeros(1, np.uint64)
    h = emul.emul_build(keep.ctypes.data, n, sigma, count.ctypes.data, br.ctypes.data, border_rows.size)
    try:
        r = O.OracleRank(bwt, sigma, "u32")
        pos = range(n + 1) if positions is None else positions
        for i in pos:
            if i < n:
                assert emul.emul_symbol_at(h, i) == bwt[i]
            for c in range(1, sigma):
                assert emul.emul_lf(h, c, i) == int(count[c]) + r.rank(c, i), (sigma, c, i)
        lay = (C.c_uint32 * 6)()
        emul.emul_layout(h, lay)
        return list(lay)
    finally:
        emul.emul_free(h)


@settings(max_examples=40, **SETTINGS)
@given(data=st.data())
def test_record_arithmetic_equals_oracle_rank(emul, data):
    sigma = data.draw(st.sampled_from([2, 3, 4, 5, 6, 7, 8, 9, 16, 17, 21, 27, 33, 64, 100, 129, 256]))
    n = data.draw(st.sampled_from([0, 1, 63, 64, 65, 127, 128, 129, 500]))
    rng = np.random.default_rng(data.draw(st.integers(0, 2 ** 32)))
    bwt = rng.integers(0, sigma, n, dtype=np.uint16).astype(np.uint8) if sigma <= 256 else None
    lay = _check_records(emul, bwt, sigma)
    if sigma <= 6:
        assert lay[0] == 0 and lay[3] == 32 and lay[4] == 6
        assert lay[5] == (5 if sigma == 6 else 0)
    else:
        assert lay[0] == 1 and lay[4] == 7 and lay[3] % 32 == 0
    if sigma == 21:
        assert lay[3] == 128  # protein: one 128-byte line per 128 positions


def test_record_arithmetic_across_superblocks(emul):
    rng = np.random.default_rng(3)
    for sigma in (6, 21):
        n = 65536 * 2 + 777
        bwt = rng.integers(0, sigma, n).astype(np.uint8)
        bwt[60000:70000] = sigma - 1  # a long run over a superblock border
        pos = sorted(set(rng.integers(0, n + 1, 600).tolist() +
                         [0, 63, 64, 65535, 65536, 65537, 131071, 131072, n - 1, n]))
        _check_records(emul, bwt, sigma, pos)
    # u16 block offsets must survive a superblock made of one symbol (text_with_rank_support.rs:85-89)
    _check_records(emul, np.full(65536, 1, np.uint8), 2, [0, 1, 64, 65535, 65536])
    _check_records(emul, np.full(65536 + 64, 3, np.uint8), 6, [0, 65535, 65536, 65599, 65600])


def build_cpp_api_test(out_dir):
    exe = os.path.join(str(out_dir), "test_api")
    libdir = os.path.join(ROOT, "genedex_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_api.cpp"), "-L", libdir, "-lgenedex_b200",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    return exe


def test_cpp_mirror_compiles_and_links(tmp_path):
    # include/genedex_b200.hpp mirrors the crate's interface for C++ hosts; it must compile against
    # the header and link against the library (running it needs a GPU: tests/test_gpu_parity.py)
    assert os.path.exists(build_cpp_api_test(tmp_path))


def test_c_abi_argument_errors_never_crash(gdx):
    """Return codes instead of unwinding across the FFI (SURVEY 8b): argument errors are reported before
    any device work, so they can be checked without a GPU."""
    L = gdx._lib
    lib = L.load()
    h = C.c_void_p()
    alph = gdx.index._alphabet_struct(gdx.alphabet.ascii_dna())
    cfg = L.gdx_config(L.GDX_I32, 4, 0, 1, L.GDX_CONSTRUCT_HOST, -1, 0)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)
    offs = np.array([0, 4], dtype=np.uint64)
    assert lib.gdx_index_build(text.ctypes.data, offs.ctypes.data, 1, C.byref(alph), C.byref(cfg), None) == L.GDX_ERR_BAD_ARG
    assert lib.gdx_index_build(text.ctypes.data, offs.ctypes.data, 0, C.byref(alph), C.byref(cfg), C.byref(h)) == L.GDX_ERR_BAD_ARG
    assert b"at least one text" in lib.gdx_last_error_message()
    cfg0 = L.gdx_config(L.GDX_I32, 0, 0, 1, L.GDX_CONSTRUCT_HOST, -1, 0)  # config.rs:28
    assert lib.gdx_index_build(text.ctypes.data, offs.ctypes.data, 1, C.byref(alph), C.byref(cfg0), C.byref(h)) == L.GDX_ERR_BAD_ARG
    bad = L.gdx_alphabet()
    bad.num_dense_symbols, bad.num_searchable_dense_symbols = 1, 1  # alphabet.rs:166-170
    assert lib.gdx_index_build(text.ctypes.data, offs.ctypes.data, 1, C.byref(bad), C.byref(cfg), C.byref(h)) == L.GDX_ERR_BAD_ARG
    q = L.gdx_queries(text.ctypes.data, None, 2, 2)
    out = np.zeros(2, dtype=np.uint64)
    assert lib.gdx_count_many(None, C.byref(q), out.ctypes.data) == L.GDX_ERR_BAD_ARG
    assert lib.gdx_get_stats(None) == L.GDX_ERR_BAD_ARG
    assert lib.gdx_index_get_info(None, None) == L.GDX_ERR_BAD_ARG
    hdr = (C.c_uint8 * lib.gdx_index_header_bytes())()
    assert lib.gdx_index_adopt_image(hdr, C.c_void_p(4096), -1, 0, C.byref(h)) == L.GDX_ERR_BAD_ARG  # bad magic
    lib.gdx_index_destroy(None)  # no-op
    lib.gdx_free_hits(None, None)


def test_c_example_compiles(tmp_path):
    # examples/basic_usage.c: the crate's basic_usage example in plain C against the header
    libdir = os.path.join(ROOT, "genedex_b200", "csrc")
    exe = str(tmp_path / "basic_usage")
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "basic_usage.c"), "-L", libdir, "-lgenedex_b200",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    assert os.path.exists(exe)


def test_concat_texts_equals_oracle_also_multithreaded(gdx):
    # construction/mod.rs:255-336; above 4 M symbols the translation runs on several host threads
    lib = gdx._lib.load()
    rng = np.random.default_rng(8)
    for total, ntexts in ((1000, 7), (6_000_000, 40)):
        cuts = np.sort(rng.integers(0, total, ntexts - 1))
        cuts[:3] = cuts[3]  # a few empty texts
        cuts = np.sort(cuts)
        io = np.frombuffer(b"ACGTNacgtn", dtype=np.uint8)[rng.integers(0, 10, total)]
        offs = np.concatenate([[0], cuts, [total]]).astype(np.uint64)
        texts = [io[int(a):int(b)].tobytes() for a, b in zip(offs[:-1], offs[1:])]
        oa = O.ALPHABETS["ascii_dna_with_n"]()
        alph = gdx.index._alphabet_struct(gdx.alphabet.ascii_dna_with_n())
        dense = np.zeros(total + ntexts, dtype=np.uint8)
        sent = np.zeros(ntexts, dtype=np.uint64)
        count = np.zeros(7, dtype=np.uint64)
        assert lib.gdx_concat_texts(io.ctypes.data, offs.ctypes.data, ntexts, C.byref(alph), dense.ctypes.data,
                                    sent.ctypes.data, count.ctypes.data) == 0
        # independent restatement with numpy
        want = np.zeros(total + ntexts, dtype=np.uint8)
        table = oa.io_to_dense
        pos = 0
        want_sent = []
        for t in texts:
            want[pos:pos + len(t)] = table[np.frombuffer(t, dtype=np.uint8)]
            pos += len(t)
            want_sent.append(pos)
            pos += 1
        assert np.array_equal(dense, want) and sent.tolist() == want_sent
        freq = np.bincount(want, minlength=7).astype(np.uint64)
        assert count.tolist() == np.concatenate([[0], np.cumsum(freq[:6])]).tolist()
        if total <= 1000:  # and the oracle agrees (small case only: the oracle also builds a suffix array)
            oidx = O.OracleIndex.build(texts, oa, "u32")
            assert np.array_equal(oidx.dense_text(), dense) and oidx.count_array().tolist() == count.tolist()
    bad = np.frombuffer(b"ACGTXACGT", dtype=np.uint8)
    offs = np.array([0, 4, 9], dtype=np.uint64)
    assert lib.gdx_concat_texts(bad.ctypes.data, offs.ctypes.data, 2, C.byref(alph), dense.ctypes.data, sent.ctypes.data,
                                count.ctypes.data) == gdx._lib.GDX_ERR_INVALID_SYMBOL
    assert lib.gdx_last_error_query() == 1


# ---- host packer (genedex_b200/csrc/host_pack.cpp): the stage that cuts the PCIe bytes of a batch to a quarter ----
def _pack_reference(alphabet, data):
    """numpy restatement: code = dense - 1 for searchable symbols, exceptions elsewhere (packed as 0)."""
    tab = np.frombuffer(bytes(alphabet.io_to_dense_table), dtype=np.uint8)
    ns = alphabet.num_searchable_dense_symbols()
    dense = tab[data]
    ok = (dense >= 1) & (dense <= ns)
    code = np.where(ok, dense - 1, 0).astype(np.uint8)
    pad = (-code.size) % 4
    code = np.concatenate([code, np.zeros(pad, dtype=np.uint8)]).reshape(-1, 4)
    packed = code[:, 0] | (code[:, 1] << 2) | (code[:, 2] << 4) | (code[:, 3] << 6)
    return packed.astype(np.uint8), np.flatnonzero(~ok).astype(np.uint64)


def _pack_library(gdx, alphabet, data):
    from genedex_b200.index import _alphabet_struct
    lib = gdx._lib.load()
    a = _alphabet_struct(alphabet)
    out = np.full((data.size + 3) // 4 + 8, 0xEE, dtype=np.uint8)
    exc = np.zeros(max(data.size, 1), dtype=np.uint64)
    n_exc = C.c_uint64()
    rc = lib.gdx_pack_symbols(C.byref(a), data.ctypes.data, data.size, out.ctypes.data, exc.ctypes.data, exc.size,
                              C.byref(n_exc))
    assert rc == 0, lib.gdx_last_error_message()
    assert np.all(out[(data.size + 3) // 4:] == 0xEE), "the packer wrote past its output"
    return out[: (data.size + 3) // 4], exc[: n_exc.value]


@pytest.mark.parametrize("size", [0, 1, 3, 4, 5, 31, 32, 33, 63, 64, 65, 1000, 262_144, 262_147, 3_000_001])
def test_pack_symbols_matches_numpy(size):
    import genedex_b200 as gdx
    rng = np.random.default_rng(size)
    for name in ("ascii_dna", "ascii_dna_with_n"):
        alphabet = getattr(gdx.alphabet, name)()
        clean = np.frombuffer(b"ACGTacgt", dtype=np.uint8)[rng.integers(0, 8, size)]
        dirty = clean.copy()
        if size:
            bad = rng.integers(0, size, max(1, size // 50))
            dirty[bad] = rng.integers(0, 256, bad.size).astype(np.uint8)
        for data in (clean, dirty, rng.integers(0, 256, size).astype(np.uint8)):
            want, want_exc = _pack_reference(alphabet, data)
            got, got_exc = _pack_library(gdx, alphabet, np.ascontiguousarray(data))
            assert np.array_equal(got, want)
            assert np.array_equal(got_exc, want_exc)


def test_pack_symbols_alphabets_without_a_nibble_split():
    """searchable bytes whose code is not a function of the low nibble take the scalar packer; more than four
    searchable symbols are refused."""
    import genedex_b200 as gdx
    lib = gdx._lib.load()
    rng = np.random.default_rng(5)
    odd = gdx.alphabet.Alphabet.from_io_symbols(bytes([0x11, 0x21, 0x31, 0x41]), 0)  # same low nibble, four codes
    data = np.array([0x11, 0x21, 0x31, 0x41, 0x51, 0x01], dtype=np.uint8)[rng.integers(0, 6, 100_003)]
    want, want_exc = _pack_reference(odd, data)
    got, got_exc = _pack_library(gdx, odd, np.ascontiguousarray(data))
    assert np.array_equal(got, want) and np.array_equal(got_exc, want_exc)
    from genedex_b200.index import _alphabet_struct
    a = _alphabet_struct(gdx.alphabet.ascii_amino_acid())
    out = np.zeros(16, dtype=np.uint8)
    n_exc = C.c_uint64()
    assert lib.gdx_pack_symbols(C.byref(a), out.ctypes.data, 4, out.ctypes.data, None, 0, C.byref(n_exc)) \
        == gdx._lib.GDX_ERR_UNSUPPORTED


def test_host_pool_runs_concurrent_jobs():
    """several host threads submit staging jobs at once (a sharded call has one per GPU): every job sees only its
    own pieces (ADVICE r1: the old pool could hand a piece of the next job to a worker leaving the previous one)"""
    import threading

    import genedex_b200 as gdx
    alphabet = gdx.alphabet.ascii_dna()
    rng = np.random.default_rng(11)
    datas = [np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)].copy()
             for n in (5_000_000, 700_001, 3_000_000, 1_500_003)]
    wants = [_pack_reference(alphabet, d)[0] for d in datas]
    errors = []

    def worker(i):
        try:
            for _ in range(6):
                got, exc = _pack_library(gdx, alphabet, datas[i])
                assert exc.size == 0 and np.array_equal(got, wants[i])
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(datas))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


def test_shard_range_is_contiguous_and_balanced():
    import genedex_b200 as gdx
    lib = gdx._lib.load()
    for n in (0, 1, 7, 8, 1001, 60_000_000, 2 ** 40 + 3):
        for world in (1, 2, 3, 4, 8):
            prev_end, sizes = 0, []
            for r in range(world):
                b, e = C.c_uint64(), C.c_uint64()
                lib.gdx_shard_range(n, r, world, C.byref(b), C.byref(e))
                assert b.value == prev_end
                prev_end = e.value
                sizes.append(e.value - b.value)
            assert prev_end == n and max(sizes) - min(sizes) <= 1


def test_rust_binding_is_generated_from_the_header():
    """rust/src/gpu/ffi.rs (the reference-side `extern "C"` block of INTEGRATION.md) is generated from
    include/genedex_b200.h: the file on disk must be the generator's output and name every exported symbol."""
    import genedex_b200 as gdx
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_rust_ffi.py"), "--check"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    rust = open(os.path.join(ROOT, "rust", "src", "gpu", "ffi.rs")).read()
    declared_in_rust = set(re.findall(r"pub fn (gdx_\w+)\(", rust))
    assert declared_in_rust == set(gdx._lib.PROTOTYPES), declared_in_rust ^ set(gdx._lib.PROTOTYPES)
    # the wrapper module only calls functions the binding declares
    used = set(re.findall(r"ffi::(gdx_\w+)\(", open(os.path.join(ROOT, "rust", "src", "gpu", "mod.rs")).read()))
    assert used and used <= declared_in_rust
    integ = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert set(re.findall(r"ffi::(gdx_\w+)\(", integ)) <= declared_in_rust


def test_bad_arguments_return_codes_instead_of_crashing():
    """ADVICE r1: nothing may unwind (or abort) across the C boundary; inconsistent sizes are GDX_ERR_BAD_ARG"""
    import genedex_b200 as gdx
    from genedex_b200.index import _alphabet_struct
    lib = gdx._lib.load()
    a = _alphabet_struct(gdx.alphabet.ascii_dna())
    text = np.frombuffer(b"ACGTACGT", dtype=np.uint8)
    bad_off = np.array([0, 8, 3], dtype=np.uint64)  # decreasing
    dense, sent, cnt = np.zeros(64, dtype=np.uint8), np.zeros(4, dtype=np.uint64), np.zeros(8, dtype=np.uint64)
    rc = lib.gdx_concat_texts(text.ctypes.data, bad_off.ctypes.data, 2, C.byref(a), dense.ctypes.data, sent.ctypes.data,
                              cnt.ctypes.data)
    assert rc == gdx._lib.GDX_ERR_BAD_ARG and b"non-decreasing" in lib.gdx_last_error_message()
    cfg = gdx._lib.gdx_config(1, 4, 0, 1, 2, -1, 0, 0)
    h = C.c_void_p()
    assert lib.gdx_index_build(text.ctypes.data, bad_off.ctypes.data, 2, C.byref(a), C.byref(cfg), C.byref(h)) \
        in (gdx._lib.GDX_ERR_BAD_ARG, gdx._lib.GDX_ERR_CUDA)
    # a corrupt image header is refused before anything is allocated from it (no device needed to find out)
    hdr = (C.c_uint8 * lib.gdx_index_header_bytes())()
    assert lib.gdx_index_adopt_image(hdr, C.c_void_p(16), -1, 0, C.byref(h)) == gdx._lib.GDX_ERR_BAD_ARG


# ---- row context table + 2-bit coded byte queries, emulated on the host (row_context.h) ------------------
def _ctx_lib(emul):
    emul.emul_ctx_entry.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    emul.emul_code_query.restype = C.c_int
    emul.emul_code_query.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    emul.emul_ctx_matches.restype = C.c_int
    emul.emul_ctx_matches.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64]
    emul.emul_ctx_valid_len.restype = C.c_uint32
    emul.emul_ctx_valid_len.argtypes = [C.c_void_p]
    return emul


def _check_row_context_entries(lib, io_to_dense, ns, dense_to_io, text, rng):
    """emul_ctx_entry / emul_code_query / emul_ctx_matches at every SA value of the first 120 and at 400 random ones,
    against a symbol-by-symbol model.  dense_to_io[d] = an IO byte of searchable symbol d."""
    entry = (C.c_uint32 * 4)()
    lo, hi = C.c_uint64(), C.c_uint64()
    searchable_io = [dense_to_io[d] for d in range(1, ns + 1)]
    checked = 0
    for at in list(range(0, 120)) + rng.integers(0, text.size, 400).tolist():
        lib.emul_ctx_entry(text.ctypes.data, at, ns, entry)
        assert entry[0] == at
        # model of vl: searchable symbols directly in front of `at`, capped at 45
        vl = 0
        while vl < 45 and at - vl - 1 >= 0 and 1 <= text[at - vl - 1] <= ns:
            vl += 1
        assert lib.emul_ctx_valid_len(entry) == vl, at
        for pos in range(1, vl + 1):
            want = text[at - pos:at]
            for variant in range(3):
                q = want.copy()
                if variant == 1:
                    j = int(rng.integers(0, pos))
                    q[j] = (q[j] % ns) + 1         # a different searchable symbol at one place (none if ns == 1)
                elif variant == 2 and pos > 1:
                    q[0] = (q[0] % ns) + 1         # the leftmost compared symbol (the last one the search reaches)
                io = bytes(dense_to_io[int(c)] for c in q)
                # the query may be longer than pos: the symbols right of pos were matched by the search already
                extra = bytes(rng.choice(searchable_io) for _ in range(int(rng.integers(0, 64 - pos + 1))))
                whole = np.frombuffer(io + extra, dtype=np.uint8)
                mis = int(rng.integers(0, 4))
                ok = lib.emul_code_query(io_to_dense.ctypes.data, ns, whole.ctypes.data, whole.size, mis,
                                         int(rng.integers(0, 2 ** 31)), C.byref(lo), C.byref(hi))
                assert ok == 1
                got = lib.emul_ctx_matches(entry, pos, lo.value, hi.value)
                assert got == int(np.array_equal(q, want)), (at, pos, variant)
                checked += 1
    return checked


def _check_staged_coding(lib, io_to_dense, ns, letters, bad_bytes, rng):
    """codes_from_staged for every length 1..64 and misalignment; letters = IO bytes of searchable symbols"""
    lo, hi = C.c_uint64(), C.c_uint64()
    for tail in range(1, 65):
        for mis in range(4):
            q = letters[rng.integers(0, letters.size, tail)].copy()
            ok = lib.emul_code_query(io_to_dense.ctypes.data, ns, q.ctypes.data, tail, mis, int(rng.integers(0, 2 ** 31)),
                                     C.byref(lo), C.byref(hi))
            assert ok == 1
            value = lo.value | (hi.value << 64)
            want = sum((int(io_to_dense[b]) - 1) << (2 * j) for j, b in enumerate(q.tolist()))
            assert value == want, (tail, mis)          # also: nothing set above the last symbol
            for bad in bad_bytes:
                q2 = q.copy()
                q2[int(rng.integers(0, tail))] = bad
                assert lib.emul_code_query(io_to_dense.ctypes.data, ns, q2.ctypes.data, tail, mis, 7,
                                           C.byref(lo), C.byref(hi)) == 0, (tail, mis, bad)


def _wide_io_table(rng, ns):
    """IO byte -> dense symbol of a 256-symbol alphabet with ns searchable symbols: three IO bytes per searchable
    symbol, eight invalid bytes, every other byte a symbol above ns.  -> (io_to_dense, dense_to_io)"""
    perm = rng.permutation(256)
    io_to_dense = rng.integers(ns + 1, 256, 256).astype(np.uint8)
    for k, b in enumerate(perm[: 3 * ns]):
        io_to_dense[b] = k % ns + 1
    io_to_dense[perm[3 * ns: 3 * ns + 8]] = 0
    return io_to_dense, {d: int(perm[d - 1]) for d in range(1, ns + 1)}


def test_row_context_entry_and_comparison_equal_a_plain_model(emul):
    """The verification the kernel does from one 16-byte entry must say exactly what a symbol-by-symbol comparison of
    query[0..pos) with the text in front of SA[row] says, whenever the entry claims to cover pos symbols."""
    lib = _ctx_lib(emul)
    rng = np.random.default_rng(12)
    oa = O.ALPHABETS["ascii_dna_with_n"]()
    io_to_dense = np.array(oa.io_to_dense, dtype=np.uint8)
    ns = oa.num_searchable
    # dense text: texts of many lengths separated by sentinels (0), N (5) sprinkled in runs
    pieces = []
    for m in (1, 2, 3, 44, 45, 46, 47, 90, 200, 1000):
        t = rng.integers(1, 5, m, dtype=np.uint8)
        if m >= 90:
            for s in rng.integers(0, m - 3, 3):
                t[s:s + int(rng.integers(1, 4))] = 5
        pieces += [t, np.zeros(1, np.uint8)]
    text = np.concatenate(pieces)
    dense_to_io = {1: ord("A"), 2: ord("C"), 3: ord("G"), 4: ord("T"), 5: ord("N")}
    assert _check_row_context_entries(lib, io_to_dense, ns, dense_to_io, text, rng) > 20_000


@pytest.mark.parametrize("ns", [1, 2, 3, 4])
def test_row_context_entries_over_wide_dense_texts(emul, ns):
    """The same for alphabets with 1..4 searchable symbols among 256 dense ones (the generic rank layout with 8-bit
    text keeps the table on): every symbol above ns, whatever its value, must end the entry's context."""
    lib = _ctx_lib(emul)
    rng = np.random.default_rng(40 + ns)
    io_to_dense, dense_to_io = _wide_io_table(rng, ns)
    pieces = []
    for m in (1, 2, 3, 44, 45, 46, 47, 90, 200, 1000):
        t = rng.integers(1, ns + 1, m, dtype=np.uint8)
        if m >= 44:
            for s in rng.integers(0, m - 3, 1 + m // 60):
                t[s:s + int(rng.integers(1, 4))] = rng.choice([ns + 1, 127, 128, 250, 255])  # also: the top bit set
        pieces += [t, np.zeros(1, np.uint8)]
    text = np.concatenate(pieces)
    assert _check_row_context_entries(lib, io_to_dense, ns, dense_to_io, text, rng) > 5_000


def test_coding_of_staged_byte_queries(emul):
    """codes_from_staged: every length 1..64, every misalignment, garbage around the query in the slot; a byte that
    is not a searchable symbol (N, lower-case n, an invalid byte) anywhere in the query makes it return false."""
    lib = _ctx_lib(emul)
    rng = np.random.default_rng(4)
    oa = O.ALPHABETS["ascii_dna_with_n"]()
    io_to_dense = np.array(oa.io_to_dense, dtype=np.uint8)
    _check_staged_coding(lib, io_to_dense, oa.num_searchable, np.frombuffer(b"ACGTacgt", dtype=np.uint8),
                         (ord("N"), ord("n"), ord("x"), 0, 255), rng)


@pytest.mark.parametrize("ns", [1, 2, 3, 4])
def test_coding_of_staged_byte_queries_for_every_small_ns(emul, ns):
    """The same with 1..4 searchable symbols, where most IO bytes are valid symbols that are not searchable"""
    lib = _ctx_lib(emul)
    rng = np.random.default_rng(70 + ns)
    io_to_dense, _ = _wide_io_table(rng, ns)
    letters = np.flatnonzero((io_to_dense >= 1) & (io_to_dense <= ns)).astype(np.uint8)
    others = np.flatnonzero((io_to_dense == 0) | (io_to_dense > ns))
    assert letters.size == 3 * ns and others.size == 256 - 3 * ns
    bad = [int(b) for b in np.flatnonzero(io_to_dense == 0)[:2]] + [int(b) for b in rng.choice(others, 6, replace=False)]
    _check_staged_coding(lib, io_to_dense, ns, letters, bad, rng)


def test_check_of_prepacked_codes_equals_a_plain_model(emul):
    """packed_codes_unsearchable (k_search with a caller's 2-bit batch): true iff one of the first nsym codes is >= ns;
    codes past nsym (the next query of the stream) are never looked at; always false with 4 searchable symbols."""
    emul.emul_packed_unsearchable.restype = C.c_int
    emul.emul_packed_unsearchable.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
    rng = np.random.default_rng(5)
    for ns in (1, 2, 3, 4):
        for nsym in range(0, 65):
            for _ in range(12):
                codes = rng.integers(0, ns, 64)
                codes[nsym:] = rng.integers(0, 4, 64 - nsym)          # anything behind the query
                if nsym and rng.random() < 0.6:
                    codes[int(rng.integers(0, nsym))] = int(rng.integers(0, 4))
                v = sum(int(c) << (2 * j) for j, c in enumerate(codes))
                want = int(any(int(c) >= ns for c in codes[:nsym]))
                got = emul.emul_packed_unsearchable(v & (2 ** 64 - 1), v >> 64, nsym, ns)
                assert got == want, (ns, nsym, codes.tolist())
