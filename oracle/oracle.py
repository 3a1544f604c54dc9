"""ctypes binding of the CPU oracle (oracle/gdx_oracle.c) plus a naive pure-Python search.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs, never by the product package `genedex_b200`.  See oracle/gdx_oracle.h for the parity status
and the reference citations (all file:line are relative to /root/reference).
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile
from typing import Iterable, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libgdx_oracle.so")

I32, U32, I64 = 0, 1, 2
STORAGE = {"i32": I32, "u32": U32, "i64": I64}

OK = 0
PANIC_INVALID_SYMBOL = 1
PANIC_LOOKUP_OOB = 2
PANIC_TEXT_TOO_LONG = 3
PANIC_BAD_CONFIG = 4


class OraclePanic(RuntimeError):
    """Models a panic of the reference (the code says which one)."""

    def __init__(self, code: int, query: int | None = None):
        self.code = code
        self.query = query
        super().__init__(f"oracle: reference would panic (code {code}, query {query})")


def build_library(force: bool = False) -> str:
    """Portable build by default (the .so travels between machines).  With GDX_ORACLE_NATIVE=1 (set by
    bench.py for the CPU-baseline legs) a -march=native library is built on the machine it runs on, into a
    fresh temporary directory: the tree may be read-only, and a native build must not travel."""
    src = os.path.join(_HERE, "gdx_oracle.c")
    newest = max(os.path.getmtime(src), os.path.getmtime(os.path.join(_HERE, "gdx_oracle.h")))
    if os.environ.get("GDX_ORACLE_NATIVE") == "1":
        out = tempfile.mkdtemp(prefix="gdx_oracle_native_")
        try:
            subprocess.check_call(["make", "-C", _HERE, "-s", "native", "OUT=" + out], stdout=sys.stderr)
            return os.path.join(out, "libgdx_oracle_native.so")
        except Exception:
            shutil.rmtree(out, ignore_errors=True)  # no compiler on this machine: fall back to the portable build
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < newest:
        subprocess.check_call(["make", "-C", _HERE, "-s"], stdout=sys.stderr)
    return _LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        path = build_library()
        L = C.CDLL(path)
        if path != _LIB_PATH:  # a native build in its temporary directory: loaded, nothing left to keep
            shutil.rmtree(os.path.dirname(path), ignore_errors=True)
        u8p, u16p, u64p, i64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint16, C.c_uint64, C.c_int64))
        vp = C.c_void_p
        L.gdxo_build.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                 C.c_int, C.POINTER(vp)]
        L.gdxo_from_parts.argtypes = [vp, C.c_uint64, vp, C.c_uint32, C.c_uint32, vp, vp, C.c_uint64, vp,
                                      C.c_uint64, C.c_uint32, vp, vp, C.c_uint64, C.c_uint32, C.c_int,
                                      C.c_int, C.POINTER(vp)]
        L.gdxo_free.argtypes = [vp]
        for name, res in [("gdxo_text_len", C.c_uint64), ("gdxo_num_texts", C.c_uint64),
                          ("gdxo_dense_text", u8p), ("gdxo_suffix_array", i64p), ("gdxo_bwt", u8p),
                          ("gdxo_count_array", u64p), ("gdxo_sentinel_indices", u64p),
                          ("gdxo_frequency_table", u64p), ("gdxo_num_border", C.c_uint64),
                          ("gdxo_border_rows", u64p), ("gdxo_border_pos", u64p),
                          ("gdxo_num_samples", C.c_uint64), ("gdxo_num_superblock_offsets", C.c_uint64)]:
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = res
        L.gdxo_sample.argtypes = [vp, C.c_uint64]
        L.gdxo_sample.restype = C.c_uint64
        L.gdxo_blocks.argtypes = [vp, u64p]
        L.gdxo_blocks.restype = u64p
        L.gdxo_block_offsets.argtypes = [vp, u64p]
        L.gdxo_block_offsets.restype = u16p
        L.gdxo_superblock_offset.argtypes = [vp, C.c_uint64]
        L.gdxo_superblock_offset.restype = C.c_uint64
        L.gdxo_lookup_table_len.argtypes = [vp, C.c_uint32]
        L.gdxo_lookup_table_len.restype = C.c_uint64
        L.gdxo_lookup_entry.argtypes = [vp, C.c_uint32, C.c_uint64, u64p, u64p]
        L.gdxo_rank_construct.argtypes = [vp, C.c_uint64, C.c_uint32, C.c_int]
        L.gdxo_rank_construct.restype = vp
        L.gdxo_rank_free.argtypes = [vp]
        L.gdxo_rank_query.argtypes = [vp, C.c_uint8, C.c_uint64]
        L.gdxo_rank_query.restype = C.c_uint64
        L.gdxo_rank_symbol_at.argtypes = [vp, C.c_uint64]
        L.gdxo_rank_symbol_at.restype = C.c_uint8
        L.gdxo_rank_batch.argtypes = [vp, vp, vp, vp, C.c_uint32]
        L.gdxo_vrank_construct.argtypes = [vp, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_uint32]
        L.gdxo_vrank_construct.restype = vp
        L.gdxo_vrank_free.argtypes = [vp]
        L.gdxo_vrank_query.argtypes = [vp, C.c_uint8, C.c_uint64]
        L.gdxo_vrank_query.restype = C.c_uint64
        L.gdxo_vrank_symbol_at.argtypes = [vp, C.c_uint64]
        L.gdxo_vrank_symbol_at.restype = C.c_uint8
        L.gdxo_vrank_blocks.argtypes = [vp, u64p]
        L.gdxo_vrank_blocks.restype = u64p
        L.gdxo_vrank_block_offsets.argtypes = [vp, u64p]
        L.gdxo_vrank_block_offsets.restype = u16p
        for name in ("gdxo_vrank_num_superblock_offsets", "gdxo_vrank_superblock_size"):
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = C.c_uint64
        L.gdxo_vrank_superblock_offset.argtypes = [vp, C.c_uint64]
        L.gdxo_vrank_superblock_offset.restype = C.c_uint64
        L.gdxo_tree_lookup.argtypes = [vp, C.c_uint64, C.c_uint64]
        L.gdxo_tree_lookup.restype = C.c_uint64
        L.gdxo_cursor_for_query.argtypes = [vp, vp, C.c_uint64, u64p, u64p]
        L.gdxo_extend_query_front.argtypes = [vp, C.c_uint8, u64p, u64p]
        L.gdxo_cursors_many.argtypes = [vp, vp, vp, C.c_uint64, vp, vp, u64p]
        L.gdxo_count_many.argtypes = [vp, vp, vp, C.c_uint64, C.c_int, vp, u64p]
        L.gdxo_locate_interval.argtypes = [vp, C.c_uint64, C.c_uint64, vp]
        L.gdxo_locate_many.argtypes = [vp, vp, vp, C.c_uint64, C.c_int, vp, C.POINTER(vp), u64p]
        L.gdxo_free_hits.argtypes = [vp]
        L.gdxo_online_cores.restype = C.c_int
        L.gdxo_verify_against_text.argtypes = [vp, vp, C.c_uint64, C.c_int, u64p, u64p]
        _lib = L
    return _lib


# ---- alphabets (alphabet.rs:43-149, 251-345) -----------------------------------------------------

class OracleAlphabet:
    """io_to_dense table + sizes; dense 0 is the sentinel (alphabet.rs:14-16)."""

    def __init__(self, groups: Sequence[bytes], num_not_searchable: int = 0):
        table = np.zeros(256, dtype=np.uint8)
        seen = set()
        assert 1 <= len(groups) <= 255
        for i, g in enumerate(groups):
            assert len(g) > 0
            for s in g:
                assert s not in seen, "Symbols of the alphabet must be unique."
                seen.add(s)
                table[s] = i + 1
        self.io_to_dense = table
        self.dense_to_io = bytes(g[0] for g in groups)
        self.sigma = len(groups) + 1
        self.num_searchable = self.sigma - num_not_searchable - 1
        assert num_not_searchable + 2 <= self.sigma


def _groups(*gs: bytes):
    return list(gs)


ALPHABETS = {
    "ascii_dna": lambda: OracleAlphabet(_groups(b"Aa", b"Cc", b"Gg", b"Tt"), 0),
    "ascii_dna_with_n": lambda: OracleAlphabet(_groups(b"Aa", b"Cc", b"Gg", b"Tt", b"Nn"), 1),
    "ascii_dna_iupac": lambda: OracleAlphabet(
        _groups(b"Aa", b"Cc", b"Gg", b"Tt", b"Nn", b"Rr", b"Yy", b"Kk", b"Mm", b"Ss", b"Ww", b"Bb", b"Dd",
                b"Hh", b"Vv"), 0),
    "ascii_dna_iupac_as_dna_with_n": lambda: OracleAlphabet(
        _groups(b"Aa", b"Cc", b"Gg", b"Tt", b"NnRrYyKkMmSsWwBbDdHhVv"), 1),
    "ascii_amino_acid": lambda: OracleAlphabet(
        [bytes([c, c + 32]) for c in b"ACDEFGHIKLMNOPQRSTUVWY"], 0),
    "ascii_amino_acid_iupac": lambda: OracleAlphabet(
        [bytes([c, c + 32]) for c in b"ABCDEFGHIJKLMNOPQRSTUVWXYZ"] + [b"*"], 0),
    "ascii_printable": lambda: OracleAlphabet([bytes([c]) for c in range(32, 127)], 0),
    "protein20": lambda: OracleAlphabet([bytes([c]) for c in b"ACDEFGHIKLMNPQRSTVWY"], 0),
}


def u8_until(max_symbol: int) -> OracleAlphabet:
    return OracleAlphabet([bytes([c]) for c in range(0, max_symbol + 1)], 0)


# ---- helpers -------------------------------------------------------------------------------------

def pack(seqs: Iterable[bytes | Sequence[int]]):
    """Concatenate sequences into (bytes array, offsets[nq+1] uint64)."""
    seqs = [bytes(s) for s in seqs]
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    if seqs:
        offsets[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    data = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy() if seqs else np.zeros(0, np.uint8)
    if data.size == 0:
        data = np.zeros(1, dtype=np.uint8)  # keep a valid pointer
    return data, offsets


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _check(rc: int, query: int | None = None):
    if rc != OK:
        raise OraclePanic(rc, query)


class OracleRank:
    """CondensedTextWithRankSupport<I, Block64> (condensed.rs)."""

    def __init__(self, dense_text, sigma: int, storage: str = "i32"):
        t = np.ascontiguousarray(np.asarray(dense_text, dtype=np.uint8))
        self._keep = t if t.size else np.zeros(1, np.uint8)
        self.n = int(t.size)
        self.h = lib().gdxo_rank_construct(_ptr(self._keep), self.n, sigma, STORAGE[storage])
        if not self.h:
            raise OraclePanic(PANIC_BAD_CONFIG)

    def rank(self, symbol: int, idx: int) -> int:
        return int(lib().gdxo_rank_query(self.h, symbol, idx))

    def symbol_at(self, idx: int) -> int:
        return int(lib().gdxo_rank_symbol_at(self.h, idx))

    def rank_batch(self, symbols, starts, ends):
        s = np.ascontiguousarray(symbols, dtype=np.uint8)
        a = np.ascontiguousarray(starts, dtype=np.uint64).copy()
        b = np.ascontiguousarray(ends, dtype=np.uint64).copy()
        assert len(s) <= 64
        lib().gdxo_rank_batch(self.h, _ptr(s), _ptr(a), _ptr(b), len(s))
        return a, b

    def __del__(self):
        if getattr(self, "h", None):
            lib().gdxo_rank_free(self.h)
            self.h = None


class OracleVariantRank:
    """TextWithRankSupport in any of the crate's four variants (lib.rs:104-113): variant "condensed" | "flat",
    block_bits 64 | 512, arrays in the reference's own layout."""

    def __init__(self, dense_text, sigma: int, storage: str = "i32", variant: str = "condensed", block_bits: int = 64):
        t = np.ascontiguousarray(np.asarray(dense_text, dtype=np.uint8))
        self.n, self.sigma, self.variant, self.block_bits = int(t.size), sigma, variant, block_bits
        self.h = lib().gdxo_vrank_construct(_ptr(t) if t.size else None, t.size, sigma, STORAGE[storage],
                                            0 if variant == "condensed" else 1, block_bits)
        if not self.h:
            raise ValueError("bad rank variant parameters")

    def rank(self, symbol: int, idx: int) -> int:
        return int(lib().gdxo_vrank_query(self.h, symbol, idx))

    def symbol_at(self, idx: int) -> int:
        return int(lib().gdxo_vrank_symbol_at(self.h, idx))

    def blocks(self) -> np.ndarray:
        n = C.c_uint64()
        p = lib().gdxo_vrank_blocks(self.h, C.byref(n))
        return np.ctypeslib.as_array(p, shape=(max(n.value, 1),))[: n.value].copy()

    def block_offsets(self) -> np.ndarray:
        n = C.c_uint64()
        p = lib().gdxo_vrank_block_offsets(self.h, C.byref(n))
        if not n.value:
            return np.zeros(0, dtype=np.uint16)
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy()

    def superblock_offsets(self) -> np.ndarray:
        k = int(lib().gdxo_vrank_num_superblock_offsets(self.h))
        return np.array([lib().gdxo_vrank_superblock_offset(self.h, i) for i in range(k)], dtype=np.uint64)

    def superblock_size(self) -> int:
        return int(lib().gdxo_vrank_superblock_size(self.h))

    def __del__(self):
        if getattr(self, "h", None):
            lib().gdxo_vrank_free(self.h)
            self.h = None


class OracleIndex:
    """FmIndex<I, CondensedTextWithRankSupport<I, Block64>> (lib.rs:93-100)."""

    def __init__(self, handle, alphabet: OracleAlphabet):
        self.h = handle
        self.alphabet = alphabet

    @classmethod
    def build(cls, texts: Sequence[bytes], alphabet: OracleAlphabet, storage: str = "i32",
              sampling_rate: int = 4, lookup_depth: int = 0) -> "OracleIndex":
        data, offsets = pack(texts)
        h = C.c_void_p()
        rc = lib().gdxo_build(_ptr(data), _ptr(offsets), len(texts), _ptr(alphabet.io_to_dense),
                              alphabet.sigma, alphabet.num_searchable, sampling_rate, lookup_depth,
                              STORAGE[storage], C.byref(h))
        _check(rc)
        return cls(h, alphabet)

    @classmethod
    def from_parts(cls, bwt: np.ndarray, alphabet: OracleAlphabet, count, sentinel_indices,
                   sampled_sa=None, sampling_rate: int = 4, border_rows=None, border_pos=None,
                   lookup_depth: int = 0, storage: str = "u32", nthreads: int = 0) -> "OracleIndex":
        bwt = np.ascontiguousarray(bwt, dtype=np.uint8)
        count = np.ascontiguousarray(count, dtype=np.uint64)
        sent = np.ascontiguousarray(sentinel_indices, dtype=np.uint64)
        ssa = None if sampled_sa is None else np.ascontiguousarray(sampled_sa, dtype=np.uint64)
        br = None if border_rows is None else np.ascontiguousarray(border_rows, dtype=np.uint64)
        bp = None if border_pos is None else np.ascontiguousarray(border_pos, dtype=np.uint64)
        h = C.c_void_p()
        rc = lib().gdxo_from_parts(_ptr(bwt), bwt.size, _ptr(alphabet.io_to_dense), alphabet.sigma,
                                   alphabet.num_searchable, _ptr(count), _ptr(sent), sent.size,
                                   None if ssa is None else _ptr(ssa), 0 if ssa is None else ssa.size,
                                   sampling_rate, None if br is None else _ptr(br),
                                   None if bp is None else _ptr(bp), 0 if br is None else br.size,
                                   lookup_depth, STORAGE[storage], nthreads, C.byref(h))
        _check(rc)
        return cls(h, alphabet)

    def __del__(self):
        if getattr(self, "h", None):
            lib().gdxo_free(self.h)
            self.h = None

    def verify_against_text(self, dense_text: np.ndarray, nthreads: int = 0) -> tuple[int, int]:
        """gdxo_verify_against_text -> (violations, rows visited): 0 and text_len for an index whose BWT,
        samples and border map really belong to `dense_text`."""
        t = np.ascontiguousarray(dense_text, dtype=np.uint8)
        bad, seen = C.c_uint64(), C.c_uint64()
        _check(lib().gdxo_verify_against_text(self.h, _ptr(t), t.size, nthreads, C.byref(bad), C.byref(seen)))
        return int(bad.value), int(seen.value)

    # -- introspection
    @property
    def text_len(self) -> int:
        return int(lib().gdxo_text_len(self.h))

    @property
    def num_texts(self) -> int:
        return int(lib().gdxo_num_texts(self.h))

    def _arr(self, fn, n, dtype):
        p = fn(self.h)
        if not p or n == 0:
            return np.zeros(0, dtype=dtype)
        return np.ctypeslib.as_array(p, shape=(n,)).copy()

    def dense_text(self):
        return self._arr(lib().gdxo_dense_text, self.text_len, np.uint8)

    def suffix_array(self):
        return self._arr(lib().gdxo_suffix_array, self.text_len, np.int64)

    def bwt(self):
        return self._arr(lib().gdxo_bwt, self.text_len, np.uint8)

    def count_array(self):
        return self._arr(lib().gdxo_count_array, self.alphabet.sigma + 1, np.uint64)

    def sentinel_indices(self):
        return self._arr(lib().gdxo_sentinel_indices, self.num_texts, np.uint64)

    def frequency_table(self):
        return self._arr(lib().gdxo_frequency_table, 256, np.uint64)

    def border(self):
        n = int(lib().gdxo_num_border(self.h))
        return self._arr(lib().gdxo_border_rows, n, np.uint64), self._arr(lib().gdxo_border_pos, n, np.uint64)

    def samples(self):
        n = int(lib().gdxo_num_samples(self.h))
        return np.array([lib().gdxo_sample(self.h, k) for k in range(n)], dtype=np.uint64)

    def blocks(self):
        n = C.c_uint64()
        p = lib().gdxo_blocks(self.h, C.byref(n))
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy()

    def block_offsets(self):
        n = C.c_uint64()
        p = lib().gdxo_block_offsets(self.h, C.byref(n))
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy()

    def superblock_offsets(self):
        n = int(lib().gdxo_num_superblock_offsets(self.h))
        return np.array([lib().gdxo_superblock_offset(self.h, k) for k in range(n)], dtype=np.uint64)

    def lookup_table(self, depth: int):
        n = int(lib().gdxo_lookup_table_len(self.h, depth))
        out = np.zeros((n, 2), dtype=np.uint64)
        s, e = C.c_uint64(), C.c_uint64()
        for i in range(n):
            lib().gdxo_lookup_entry(self.h, depth, i, C.byref(s), C.byref(e))
            out[i] = (s.value, e.value)
        return out

    # -- single query (lib.rs:147-149,169-173,217-235)
    def cursor_for_query(self, q: bytes):
        q = bytes(q)
        buf = np.frombuffer(q, dtype=np.uint8) if q else np.zeros(1, np.uint8)
        s, e = C.c_uint64(), C.c_uint64()
        _check(lib().gdxo_cursor_for_query(self.h, _ptr(buf), len(q), C.byref(s), C.byref(e)))
        return s.value, e.value

    def extend_query_front(self, interval, io_symbol: int):
        s, e = C.c_uint64(interval[0]), C.c_uint64(interval[1])
        _check(lib().gdxo_extend_query_front(self.h, io_symbol, C.byref(s), C.byref(e)))
        return s.value, e.value

    def count(self, q: bytes) -> int:
        s, e = self.cursor_for_query(q)
        return e - s

    def locate_interval(self, start: int, end: int):
        n = end - start
        out = np.zeros((max(n, 1), 2), dtype=np.uint64)
        _check(lib().gdxo_locate_interval(self.h, start, end, _ptr(out)))
        return [(int(t), int(p)) for t, p in out[:n]]

    def locate(self, q: bytes):
        s, e = self.cursor_for_query(q)
        return self.locate_interval(s, e)

    # -- batched (lib.rs:155-185,241-246)
    def cursors_many_packed(self, data: np.ndarray, offsets: np.ndarray):
        nq = offsets.size - 1
        starts = np.zeros(max(nq, 1), dtype=np.uint64)
        ends = np.zeros(max(nq, 1), dtype=np.uint64)
        pq = C.c_uint64()
        rc = lib().gdxo_cursors_many(self.h, _ptr(data), _ptr(offsets), nq, _ptr(starts), _ptr(ends),
                                     C.byref(pq))
        _check(rc, pq.value)
        return starts[:nq], ends[:nq]

    def cursors_many(self, queries):
        return self.cursors_many_packed(*pack(queries))

    def count_many_packed(self, data: np.ndarray, offsets: np.ndarray, nthreads: int = 1):
        nq = offsets.size - 1
        counts = np.zeros(max(nq, 1), dtype=np.uint64)
        pq = C.c_uint64()
        rc = lib().gdxo_count_many(self.h, _ptr(data), _ptr(offsets), nq, nthreads, _ptr(counts),
                                   C.byref(pq))
        _check(rc, pq.value)
        return counts[:nq]

    def count_many(self, queries, nthreads: int = 1):
        return self.count_many_packed(*pack(queries), nthreads=nthreads)

    def locate_many_packed(self, data: np.ndarray, offsets: np.ndarray, nthreads: int = 1):
        """Returns (hit_offsets[nq+1], hits[(n,2)] as (text_id, position)) in SA-row order."""
        nq = offsets.size - 1
        hit_offsets = np.zeros(nq + 1, dtype=np.uint64)
        hp = C.c_void_p()
        pq = C.c_uint64()
        rc = lib().gdxo_locate_many(self.h, _ptr(data), _ptr(offsets), nq, nthreads, _ptr(hit_offsets),
                                    C.byref(hp), C.byref(pq))
        _check(rc, pq.value)
        total = int(hit_offsets[nq])
        if total:
            buf = (C.c_uint64 * (2 * total)).from_address(hp.value)
            hits = np.frombuffer(buf, dtype=np.uint64).reshape(total, 2).copy()
        else:
            hits = np.zeros((0, 2), dtype=np.uint64)
        lib().gdxo_free_hits(hp)
        return hit_offsets, hits

    def locate_many(self, queries, nthreads: int = 1):
        off, hits = self.locate_many_packed(*pack(queries), nthreads=nthreads)
        return [[(int(t), int(p)) for t, p in hits[int(off[i]):int(off[i + 1])]]
                for i in range(len(off) - 1)]


def tree_lookup(sentinel_indices, pos: int) -> int:
    s = np.ascontiguousarray(sentinel_indices, dtype=np.uint64)
    return int(lib().gdxo_tree_lookup(_ptr(s), s.size, pos))


# ---- naive references written the way the reference's tests write them ---------------------------

def naive_search(texts: Sequence[bytes], query: bytes, fold=None):
    """tests/fmindex.rs:207-227 naive_search; `fold` maps IO bytes to a canonical form so that
    case-insensitive / ambiguous alphabets compare equal (e.g. the io_to_dense table)."""
    hits = set()
    if fold is not None:
        query = bytes(fold[b] for b in query)
    for text_id, text in enumerate(texts):
        if fold is not None:
            text = bytes(fold[b] for b in text)
        if len(query) == 0:
            for position in range(len(text) + 1):
                hits.add((text_id, position))
            continue
        start = 0
        while True:
            p = text.find(query, start)
            if p < 0:
                break
            hits.add((text_id, p))
            start = p + 1
    return hits


def naive_suffix_array(dense_text: Sequence[int]) -> list[int]:
    """Plain sort of all suffixes; a proper prefix sorts first (libsais convention)."""
    t = bytes(dense_text)
    return sorted(range(len(t)), key=lambda i: t[i:])
