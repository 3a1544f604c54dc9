"""Host-side mirror of genedex's public search interface over the C ABI (include/genedex_b200.h).

Same names, argument meaning and error behaviour as the crate (src/lib.rs, src/config.rs,
src/cursor.rs); a reference panic surfaces as a Python exception.  All compute goes through
libgenedex_b200.so on the GPU -- there is no CPU path in this package.
"""
from __future__ import annotations

import ctypes as C
import enum
import os
from dataclasses import dataclass
from typing import Iterable, Sequence

import numpy as np

from . import _lib
from .alphabet import Alphabet


class GenedexError(RuntimeError):
    def __init__(self, status: int, message: str, query: int | None = None):
        self.status = status
        self.query = query
        super().__init__(message)


class InvalidSymbolError(GenedexError, ValueError):
    """The reference panics 'symbol in io representation should be valid' (src/alphabet.rs:195-198)."""


def _check(status: int):
    if status == _lib.GDX_OK:
        return
    lib = _lib.load()
    msg = lib.gdx_last_error_message().decode("utf-8", "replace")
    if status == _lib.GDX_ERR_INVALID_SYMBOL:
        raise InvalidSymbolError(status, msg, int(lib.gdx_last_error_query()))
    if status == _lib.GDX_ERR_OOM:
        raise MemoryError(msg)
    raise GenedexError(status, msg)


class PerformancePriority(enum.IntEnum):  # src/config.rs:89-102
    HighSpeed = 0
    Balanced = 1
    LowMemory = 2


_STORAGE = {"i32": _lib.GDX_I32, "u32": _lib.GDX_U32, "i64": _lib.GDX_I64}


@dataclass(frozen=True, order=True)
class Hit:  # src/lib.rs:331-335
    text_id: int
    position: int


def pack_queries(queries: Iterable[bytes]):
    """Any iterable of bytes-like -> (uint8 array, uint64 offsets[nq+1])."""
    qs = [bytes(q) for q in queries]
    offsets = np.zeros(len(qs) + 1, dtype=np.uint64)
    if qs:
        offsets[1:] = np.cumsum([len(q) for q in qs], dtype=np.uint64)
    data = np.frombuffer(b"".join(qs), dtype=np.uint8)
    if data.size == 0:
        data = np.zeros(1, dtype=np.uint8)
    return np.ascontiguousarray(data), offsets


def _queries_struct(data: np.ndarray, offsets: np.ndarray | None, fixed_len: int, nq: int,
                    encoding: int = _lib.GDX_QUERIES_IO_BYTES) -> _lib.gdx_queries:
    return _lib.gdx_queries(data.ctypes.data, None if offsets is None else offsets.ctypes.data, fixed_len, nq,
                            encoding, 0)


class FmIndexConfig:
    """Builder, src/config.rs:9-70. `storage` plays the role of the generic parameter I."""

    def __init__(self, storage: str = "i32"):
        assert storage in _STORAGE
        self.storage = storage
        self._sampling_rate = 4          # config.rs:75
        self._lookup_depth = 0           # config.rs:76
        self._priority = PerformancePriority.Balanced  # config.rs:77
        self._construction = _lib.GDX_CONSTRUCT_AUTO  # all construction routes give the same index
        self._device = -1
        self._flags = 0
        self._accel_budget = 0

    def suffix_array_sampling_rate(self, rate: int) -> "FmIndexConfig":
        assert rate > 0  # config.rs:28
        self._sampling_rate = rate
        return self

    def lookup_table_depth(self, depth: int) -> "FmIndexConfig":
        self._lookup_depth = depth
        return self

    def construction_performance_priority(self, p: PerformancePriority) -> "FmIndexConfig":
        self._priority = p
        return self

    # -- additions of this engine (not in the reference): where to build, on which GPU
    def construct_on_device(self, on_device: bool = True, verify: bool = False) -> "FmIndexConfig":
        self._construction = _lib.GDX_CONSTRUCT_DEVICE if on_device else _lib.GDX_CONSTRUCT_HOST
        self._flags = (self._flags & ~_lib.GDX_FLAG_VERIFY_SUFFIX_ARRAY) | (
            _lib.GDX_FLAG_VERIFY_SUFFIX_ARRAY if verify else 0)
        return self

    def keep_text(self, keep: bool = True) -> "FmIndexConfig":
        """Keep the packed text in the device image (default): one-row intervals are finished by a
        text comparison in count/locate.  Without it every LF step runs; results are identical."""
        self._flags = (self._flags & ~_lib.GDX_FLAG_NO_TEXT) | (0 if keep else _lib.GDX_FLAG_NO_TEXT)
        return self

    def keep_inverse_samples(self, keep: bool = True) -> "FmIndexConfig":
        """Keep the sampled inverse suffix array (default, needs the text): cursors_for_many_queries then
        finishes one-row intervals through the text as well.  Results are identical either way."""
        self._flags = (self._flags & ~_lib.GDX_FLAG_NO_INVERSE_SAMPLES) | (
            0 if keep else _lib.GDX_FLAG_NO_INVERSE_SAMPLES)
        return self

    def dense_suffix_array(self, allow: bool = True) -> "FmIndexConfig":
        """Allow (default) or forbid the dense suffix array accelerator: SA[row] for every row, 4-8 bytes
        per symbol on top of the image, built when device memory is ample (`FmIndex.set_dense_suffix_array`
        forces it).  Resolving a row is then one load instead of an LF-walk; results are identical."""
        self._flags = (self._flags & ~_lib.GDX_FLAG_NO_DENSE_SUFFIX_ARRAY) | (
            0 if allow else _lib.GDX_FLAG_NO_DENSE_SUFFIX_ARRAY)
        return self

    def seed_table(self, allow: bool = True) -> "FmIndexConfig":
        """Allow (default) or forbid the seed table accelerator: one level of a lookup table deeper than the
        configured one (largest depth with ns^depth <= 4 * text length), built when device memory is ample
        (`FmIndex.set_seed_table_depth` forces a depth).  Results and error behaviour are identical."""
        self._flags = (self._flags & ~_lib.GDX_FLAG_NO_SEED_TABLE) | (0 if allow else _lib.GDX_FLAG_NO_SEED_TABLE)
        return self

    def row_context_table(self, allow: bool = True) -> "FmIndexConfig":
        """Allow (default) or forbid the row context table accelerator: SA[row] + the 45 text symbols in front of it in
        one 16-byte entry per row (DNA-sized alphabets, texts shorter than 2^32), built last when it fits what the other
        accelerators left (`FmIndex.set_row_context_table` forces it).  Results are identical."""
        self._flags = (self._flags & ~_lib.GDX_FLAG_NO_ROW_CONTEXT_TABLE) | (
            0 if allow else _lib.GDX_FLAG_NO_ROW_CONTEXT_TABLE)
        return self

    def accelerator_budget(self, nbytes: int) -> "FmIndexConfig":
        """Device memory the accelerators of a replica (dense suffix array, seed table) may take together;
        0 = automatic (each at most a quarter of the free memory).  Travels with the index image."""
        self._accel_budget = int(nbytes)
        return self

    def device(self, ordinal: int) -> "FmIndexConfig":
        self._device = ordinal
        return self

    def construct_index(self, texts: Iterable[bytes], alphabet: Alphabet) -> "FmIndex":  # config.rs:63-69
        return self.construct_index_packed(*pack_queries(texts), alphabet)

    def construct_index_packed(self, data: np.ndarray, offsets: np.ndarray, alphabet: Alphabet) -> "FmIndex":
        """Texts as one uint8 array + uint64 offsets[num_texts + 1] (no copies of a multi-GB text)."""
        lib = _lib.load()
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        a = _alphabet_struct(alphabet)
        cfg = _lib.gdx_config(_STORAGE[self.storage], self._sampling_rate, self._lookup_depth,
                              int(self._priority), self._construction, self._device, self._flags,
                              self._accel_budget)
        h = C.c_void_p()
        _check(lib.gdx_index_build(data.ctypes.data, offsets.ctypes.data, offsets.size - 1, C.byref(a),
                                   C.byref(cfg), C.byref(h)))
        return FmIndex(h, alphabet)


def _alphabet_struct(alphabet: Alphabet) -> _lib.gdx_alphabet:
    a = _lib.gdx_alphabet()
    C.memmove(a.io_to_dense, alphabet.io_to_dense_table, 256)
    a.num_dense_symbols = alphabet.num_dense_symbols()
    a.num_searchable_dense_symbols = alphabet.num_searchable_dense_symbols()
    return a


class FmIndex:
    """src/lib.rs:93-327 over a device-resident index."""

    def __init__(self, handle: C.c_void_p, alphabet: Alphabet, keepalive=None):
        self._h = handle
        self._alphabet = alphabet
        self._keepalive = keepalive
        self._lib = _lib.load()

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.gdx_index_destroy(h)

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    # -- accessors, lib.rs:283-294
    def alphabet(self) -> Alphabet:
        return self._alphabet

    def info(self) -> _lib.gdx_index_info:
        out = _lib.gdx_index_info()
        _check(self._lib.gdx_index_get_info(self._h, C.byref(out)))
        return out

    def set_dense_suffix_array(self, on: bool = True) -> None:
        """Build now (raises if it does not fit) or free the dense suffix array accelerator."""
        _check(self._lib.gdx_index_set_dense_suffix_array(self._h, 1 if on else 0))

    def set_seed_table_depth(self, depth: int) -> None:
        """(Re)build the seed table accelerator at this depth now (raises if it does not fit); 0 frees it."""
        _check(self._lib.gdx_index_set_seed_table_depth(self._h, int(depth)))

    def set_row_context_table(self, on: bool = True) -> None:
        """Build now (raises if it does not fit / does not apply) or free the row context table accelerator."""
        _check(self._lib.gdx_index_set_row_context_table(self._h, 1 if on else 0))

    def set_text_verification(self, on: bool = True) -> None:
        """Finish one-row intervals through the text (default) or run every LF step like the reference."""
        _check(self._lib.gdx_index_set_text_verification(self._h, 1 if on else 0))

    def num_texts(self) -> int:
        return int(self.info().num_texts)

    def total_text_len(self) -> int:
        return int(self.info().text_len)

    # -- index files, lib.rs:296-327 (own container format, not savefile-compatible: DESIGN.md)
    def save_to_file(self, filepath) -> None:
        a = self._alphabet
        blob = bytes([a._not_searchable]) + a._dense_to_io
        _check(self._lib.gdx_index_save_to_file(self._h, os.fsencode(filepath), blob, len(blob)))

    @classmethod
    def load_from_file(cls, filepath, device: int = -1) -> "FmIndex":
        lib = _lib.load()
        h, nbytes = C.c_void_p(), C.c_uint64()
        blob = (C.c_uint8 * 512)()
        _check(lib.gdx_index_load_from_file(os.fsencode(filepath), device, C.byref(h), blob, 512, C.byref(nbytes)))
        idx = cls(h, None)
        hdr = (C.c_uint8 * lib.gdx_index_header_bytes())()
        _check(lib.gdx_index_export(h, hdr, None, None))
        raw = bytes(blob[: nbytes.value])
        io_to_dense = bytes(hdr)[-256:]  # last field of the image header
        idx._alphabet = Alphabet(io_to_dense, raw[1:], raw[0])
        return idx

    # -- packed (numpy) forms: the zero-copy entry points the list forms are built on
    def cursors_many_packed(self, data: np.ndarray, offsets: np.ndarray | None = None, fixed_len: int = 0,
                            nq: int | None = None, out: tuple[np.ndarray, np.ndarray] | None = None,
                            encoding: int = _lib.GDX_QUERIES_IO_BYTES):
        """-> (starts, ends); `out` = two uint64 (or two uint32) arrays of >= nq entries to fill (e.g. pinned memory)."""
        nq = (offsets.size - 1) if offsets is not None else nq
        starts, ends = out if out is not None else (np.empty(max(nq, 1), dtype=np.uint64),
                                                    np.empty(max(nq, 1), dtype=np.uint64))
        q = _queries_struct(data, offsets, fixed_len, nq, encoding)
        fn = self._lib.gdx_cursors_many_u32 if starts.dtype == np.uint32 else self._lib.gdx_cursors_many
        _check(fn(self._h, C.byref(q), starts.ctypes.data, ends.ctypes.data))
        return starts[:nq], ends[:nq]

    def count_many_packed(self, data: np.ndarray, offsets: np.ndarray | None = None, fixed_len: int = 0,
                          nq: int | None = None, out: np.ndarray | None = None,
                          encoding: int = _lib.GDX_QUERIES_IO_BYTES) -> np.ndarray:
        """`out` may be a uint64 or a uint32 array (the latter: gdx_count_many_u32, texts < 2^32 symbols);
        encoding = GDX_QUERIES_PACKED_2BIT: `data` is a 2-bit stream made by pack_queries_2bit."""
        nq = (offsets.size - 1) if offsets is not None else nq
        counts = out if out is not None else np.empty(max(nq, 1), dtype=np.uint64)
        q = _queries_struct(data, offsets, fixed_len, nq, encoding)
        fn = self._lib.gdx_count_many_u32 if counts.dtype == np.uint32 else self._lib.gdx_count_many
        assert counts.dtype in (np.uint32, np.uint64)
        _check(fn(self._h, C.byref(q), counts.ctypes.data))
        return counts[:nq]

    def pack_queries_2bit(self, data: np.ndarray, offsets: np.ndarray | None = None, fixed_len: int = 0,
                          nq: int | None = None, out: np.ndarray | None = None):
        """IO bytes -> 2-bit stream (gdx_pack_queries); -> (packed uint8 array, index of the first query that
        cannot be packed or None)."""
        nq = (offsets.size - 1) if offsets is not None else nq
        total = int(offsets[-1]) if offsets is not None else nq * fixed_len
        nbytes = int(self._lib.gdx_packed_bytes(total))
        packed = out if out is not None else np.empty(max(nbytes, 4), dtype=np.uint8)
        first = C.c_uint64()
        q = _queries_struct(data, offsets, fixed_len, nq)
        _check(self._lib.gdx_pack_queries(self._h, C.byref(q), packed.ctypes.data, C.byref(first)))
        return packed, (None if first.value == 2 ** 64 - 1 else int(first.value))

    def locate_many_packed(self, data: np.ndarray, offsets: np.ndarray | None = None, fixed_len: int = 0,
                           nq: int | None = None, encoding: int = _lib.GDX_QUERIES_IO_BYTES):
        """-> (hit_offsets[nq+1], hits[n,2] = (text_id, position)); hits of a query in SA-row order."""
        nq = (offsets.size - 1) if offsets is not None else nq
        hit_offsets = np.empty(nq + 1, dtype=np.uint64)
        hp, nh = C.c_void_p(), C.c_uint64()
        q = _queries_struct(data, offsets, fixed_len, nq, encoding)
        _check(self._lib.gdx_locate_many(self._h, C.byref(q), hit_offsets.ctypes.data, C.byref(hp), C.byref(nh)))
        return hit_offsets, self._take_hits(hp, nh.value)

    def locate_many_view(self, data: np.ndarray, offsets: np.ndarray | None = None, fixed_len: int = 0,
                         nq: int | None = None, hit_offsets: np.ndarray | None = None):
        """Zero-copy form of locate_many_packed: -> (hit_offsets, hits view on the library's pinned
        buffer, release) -- call release() when done with the view (gdx_free_hits)."""
        nq = (offsets.size - 1) if offsets is not None else nq
        if hit_offsets is None:
            hit_offsets = np.empty(nq + 1, dtype=np.uint64)
        hp, nh = C.c_void_p(), C.c_uint64()
        q = _queries_struct(data, offsets, fixed_len, nq)
        _check(self._lib.gdx_locate_many(self._h, C.byref(q), hit_offsets.ctypes.data, C.byref(hp), C.byref(nh)))
        n = nh.value
        if n:
            buf = (C.c_uint64 * (2 * n)).from_address(hp.value)
            hits = np.frombuffer(buf, dtype=np.uint64).reshape(n, 2)
        else:
            hits = np.zeros((0, 2), dtype=np.uint64)
        return hit_offsets, hits, (lambda: self._lib.gdx_free_hits(self._h, hp))

    def locate_many_compact_view(self, data: np.ndarray, offsets: np.ndarray | None = None, fixed_len: int = 0,
                                 nq: int | None = None, hit_counts: np.ndarray | None = None,
                                 encoding: int = _lib.GDX_QUERIES_IO_BYTES):
        """gdx_locate_many_compact (texts < 2^32 symbols): -> (hit_counts uint32[nq], hits view uint32[n, 2] on the
        library's pinned buffer, release).  The CSR offsets are the prefix sums of hit_counts."""
        nq = (offsets.size - 1) if offsets is not None else nq
        if hit_counts is None:
            hit_counts = np.zeros(max(nq, 1), dtype=np.uint32)
        hp, nh = C.c_void_p(), C.c_uint64()
        q = _queries_struct(data, offsets, fixed_len, nq, encoding)
        _check(self._lib.gdx_locate_many_compact(self._h, C.byref(q), hit_counts.ctypes.data, C.byref(hp), C.byref(nh)))
        n = nh.value
        if n:
            buf = (C.c_uint32 * (2 * n)).from_address(hp.value)
            hits = np.frombuffer(buf, dtype=np.uint32).reshape(n, 2)
        else:
            hits = np.zeros((0, 2), dtype=np.uint32)
        return hit_counts[:nq], hits, (lambda: self._lib.gdx_free_hits(self._h, hp))

    def _take_hits(self, hp: C.c_void_p, n: int) -> np.ndarray:
        try:
            if n == 0:
                return np.zeros((0, 2), dtype=np.uint64)
            buf = (C.c_uint64 * (2 * n)).from_address(hp.value)
            return np.frombuffer(buf, dtype=np.uint64).reshape(n, 2).copy()
        finally:
            self._lib.gdx_free_hits(self._h, hp)

    # -- approximate search (no counterpart in the reference): up to k substitutions, semantics in genedex_b200.h
    def count_many_hamming_packed(self, data: np.ndarray, offsets: np.ndarray | None, k: int, fixed_len: int = 0,
                                  nq: int | None = None) -> np.ndarray:
        """-> uint64 array (nq, k + 1): [i, d] = occurrences of query i with exactly d mismatches."""
        nq = (offsets.size - 1) if offsets is not None else nq
        counts = np.zeros((max(nq, 1), k + 1), dtype=np.uint64)
        q = _queries_struct(data, offsets, fixed_len, nq)
        _check(self._lib.gdx_count_many_hamming(self._h, C.byref(q), k, counts.ctypes.data))
        return counts[:nq]

    def cursors_many_hamming_packed(self, data: np.ndarray, offsets: np.ndarray | None, k: int, fixed_len: int = 0,
                                    nq: int | None = None):
        """-> (interval_offsets[nq + 1], starts, ends, mismatches): the intervals of query i are the entries
        interval_offsets[i] .. interval_offsets[i + 1], sorted by start."""
        nq = (offsets.size - 1) if offsets is not None else nq
        iv_offsets = np.empty(nq + 1, dtype=np.uint64)
        ip, n = C.c_void_p(), C.c_uint64()
        q = _queries_struct(data, offsets, fixed_len, nq)
        _check(self._lib.gdx_cursors_many_hamming(self._h, C.byref(q), k, iv_offsets.ctypes.data, C.byref(ip),
                                                  C.byref(n)))
        try:
            rec = np.zeros((n.value, 3), dtype=np.uint64)
            if n.value:
                buf = (_lib.gdx_hamming_interval * n.value).from_address(ip.value)
                raw = np.frombuffer(buf, dtype=np.uint64).reshape(n.value, 3)
                rec[:, :2] = raw[:, :2]
                rec[:, 2] = raw[:, 2] & 0xFFFFFFFF
        finally:
            self._lib.gdx_free_hits(self._h, ip)
        return iv_offsets, rec[:, 0], rec[:, 1], rec[:, 2].astype(np.uint32)

    def locate_many_hamming_packed(self, data: np.ndarray, offsets: np.ndarray | None, k: int, fixed_len: int = 0,
                                   nq: int | None = None):
        """-> (hit_offsets[nq + 1], hits[n, 2] = (text_id, position)); hits of a query in ascending SA-row order."""
        nq = (offsets.size - 1) if offsets is not None else nq
        hit_offsets = np.empty(nq + 1, dtype=np.uint64)
        hp, nh = C.c_void_p(), C.c_uint64()
        q = _queries_struct(data, offsets, fixed_len, nq)
        _check(self._lib.gdx_locate_many_hamming(self._h, C.byref(q), k, hit_offsets.ctypes.data, C.byref(hp),
                                                 C.byref(nh)))
        return hit_offsets, self._take_hits(hp, nh.value)

    def count_many_hamming(self, queries: Iterable[bytes], k: int) -> np.ndarray:
        return self.count_many_hamming_packed(*pack_queries(queries), k)

    def cursors_many_hamming(self, queries: Iterable[bytes], k: int) -> list[list[tuple["Cursor", int]]]:
        off, starts, ends, mism = self.cursors_many_hamming_packed(*pack_queries(queries), k)
        return [[(Cursor(self, int(starts[j]), int(ends[j])), int(mism[j])) for j in range(int(off[i]), int(off[i + 1]))]
                for i in range(off.size - 1)]

    def locate_many_hamming(self, queries: Iterable[bytes], k: int) -> list[list[Hit]]:
        return _split_hits(*self.locate_many_hamming_packed(*pack_queries(queries), k))

    def locate_intervals_packed(self, starts: np.ndarray, ends: np.ndarray):
        starts = np.ascontiguousarray(starts, dtype=np.uint64)
        ends = np.ascontiguousarray(ends, dtype=np.uint64)
        n = starts.size
        hit_offsets = np.empty(n + 1, dtype=np.uint64)
        hp, nh = C.c_void_p(), C.c_uint64()
        _check(self._lib.gdx_locate_intervals(self._h, starts.ctypes.data, ends.ctypes.data, n,
                                              hit_offsets.ctypes.data, C.byref(hp), C.byref(nh)))
        return hit_offsets, self._take_hits(hp, nh.value)

    def extend_many_packed(self, starts: np.ndarray, ends: np.ndarray, io_symbols: np.ndarray, inplace: bool = False):
        """Batched Cursor.extend_query_front; inplace=True updates the given C-contiguous uint64 arrays (the C
        call works in place; pinned arrays avoid the staging copy), otherwise copies are extended."""
        if inplace:
            assert starts.dtype == np.uint64 and ends.dtype == np.uint64 and starts.flags.c_contiguous \
                and ends.flags.c_contiguous
        else:
            starts = np.array(starts, dtype=np.uint64, order="C")  # one copy: the C call extends in place
            ends = np.array(ends, dtype=np.uint64, order="C")
        sym = np.ascontiguousarray(io_symbols, dtype=np.uint8)
        _check(self._lib.gdx_extend_many(self._h, starts.ctypes.data, ends.ctypes.data, sym.ctypes.data, starts.size))
        return starts, ends

    def download_bwt(self) -> np.ndarray:
        out = np.empty(max(self.total_text_len(), 1), dtype=np.uint8)
        _check(self._lib.gdx_index_download_bwt(self._h, out.ctypes.data))
        return out[: self.total_text_len()]

    def download_samples(self) -> np.ndarray:
        out = np.zeros(max(int(self.info().num_samples), 1), dtype=np.uint64)
        _check(self._lib.gdx_index_download_samples(self._h, out.ctypes.data))
        return out[: int(self.info().num_samples)]

    def download_text_borders(self):
        n = int(self.info().num_text_borders)
        rows, pos = np.zeros(max(n, 1), dtype=np.uint64), np.zeros(max(n, 1), dtype=np.uint64)
        _check(self._lib.gdx_index_download_text_borders(self._h, rows.ctypes.data, pos.ctypes.data))
        return rows[:n], pos[:n]

    def count_array(self) -> np.ndarray:
        out = np.zeros(self.info().num_dense_symbols + 1, dtype=np.uint64)
        _check(self._lib.gdx_index_get_count(self._h, out.ctypes.data))
        return out

    def stats(self) -> _lib.gdx_stats:
        s = _lib.gdx_stats()
        _check(self._lib.gdx_get_stats(C.byref(s)))
        return s

    # -- the crate's API
    def count(self, query: bytes) -> int:  # lib.rs:147-149
        return self.cursor_for_query(query).count()

    def count_many(self, queries: Iterable[bytes]) -> list[int]:  # lib.rs:155-161
        data, offsets = pack_queries(queries)
        return [int(c) for c in self.count_many_packed(data, offsets)]

    def locate(self, query: bytes) -> list[Hit]:  # lib.rs:169-173
        return self.cursor_for_query(query).locate()

    def locate_many(self, queries: Iterable[bytes]) -> list[list[Hit]]:  # lib.rs:179-185
        data, offsets = pack_queries(queries)
        off, hits = self.locate_many_packed(data, offsets)
        return _split_hits(off, hits)

    def cursor_empty(self) -> "Cursor":  # lib.rs:202-210
        return Cursor(self, 0, self.total_text_len())

    def cursor_for_query(self, query: bytes) -> "Cursor":  # lib.rs:217-235
        q = bytes(query)
        buf = np.frombuffer(q, dtype=np.uint8) if q else np.zeros(1, dtype=np.uint8)
        s, e = C.c_uint64(), C.c_uint64()
        _check(self._lib.gdx_cursor_for_query(self._h, buf.ctypes.data, len(q), C.byref(s), C.byref(e)))
        return Cursor(self, s.value, e.value)

    def cursors_for_many_queries(self, queries: Iterable[bytes]) -> list["Cursor"]:  # lib.rs:241-246
        data, offsets = pack_queries(queries)
        starts, ends = self.cursors_many_packed(data, offsets)
        return [Cursor(self, int(s), int(e)) for s, e in zip(starts, ends)]

    # -- addition of this engine: batched Cursor::extend_query_front (ROADMAP.md:33)
    def extend_many(self, cursors: Sequence["Cursor"], io_symbols: bytes) -> list["Cursor"]:
        s = np.array([c.interval[0] for c in cursors], dtype=np.uint64)
        e = np.array([c.interval[1] for c in cursors], dtype=np.uint64)
        s, e = self.extend_many_packed(s, e, np.frombuffer(bytes(io_symbols), dtype=np.uint8))
        return [Cursor(self, int(a), int(b)) for a, b in zip(s, e)]


def _split_hits(off: np.ndarray, hits: np.ndarray) -> list[list[Hit]]:
    out = []
    for i in range(off.size - 1):
        a, b = int(off[i]), int(off[i + 1])
        out.append([Hit(int(t), int(p)) for t, p in hits[a:b]])
    return out


class Cursor:
    """src/cursor.rs:16-73: a half-open SA interval [start, end) of the currently searched query."""

    def __init__(self, index: FmIndex, start: int, end: int):
        self.index = index
        self.interval = (start, end)

    def extend_query_front(self, symbol: int) -> None:  # cursor.rs:34-38
        s, e = self.index.extend_many_packed(np.array([self.interval[0]], dtype=np.uint64),
                                             np.array([self.interval[1]], dtype=np.uint64),
                                             np.array([symbol], dtype=np.uint8))
        self.interval = (int(s[0]), int(e[0]))

    def count(self) -> int:  # cursor.rs:61-63
        return self.interval[1] - self.interval[0]

    def locate(self) -> list[Hit]:  # cursor.rs:71-73
        off, hits = self.index.locate_intervals_packed(np.array([self.interval[0]], dtype=np.uint64),
                                                       np.array([self.interval[1]], dtype=np.uint64))
        return [Hit(int(t), int(p)) for t, p in hits]

    def clone(self) -> "Cursor":
        return Cursor(self.index, *self.interval)
