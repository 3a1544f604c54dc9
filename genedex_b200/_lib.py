"""ctypes binding of the C ABI in include/genedex_b200.h (genedex_b200/csrc/libgenedex_b200.so).

The shared library is the product; this module only declares its prototypes.  There is no CPU
fallback: if the library has not been built, importing the package fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GENEDEX_B200_LIB selects another build of the same library (kernel experiments); default: in-tree
LIB_PATH = os.environ.get("GENEDEX_B200_LIB") or os.path.join(_HERE, "csrc", "libgenedex_b200.so")

GDX_OK, GDX_ERR_INVALID_SYMBOL, GDX_ERR_BAD_ARG, GDX_ERR_CUDA, GDX_ERR_OOM, GDX_ERR_TEXT_TOO_LONG, \
    GDX_ERR_UNSUPPORTED, GDX_ERR_BUSY = range(8)
GDX_I32, GDX_U32, GDX_I64 = 0, 1, 2
GDX_CONSTRUCT_HOST, GDX_CONSTRUCT_DEVICE, GDX_CONSTRUCT_AUTO = 0, 1, 2
GDX_FLAG_VERIFY_SUFFIX_ARRAY = 1
GDX_FLAG_NO_TEXT = 2
GDX_FLAG_NO_INVERSE_SAMPLES = 4
GDX_FLAG_NO_DENSE_SUFFIX_ARRAY = 8
GDX_FLAG_NO_SEED_TABLE = 16
GDX_FLAG_NO_ROW_CONTEXT_TABLE = 32
GDX_QUERIES_IO_BYTES, GDX_QUERIES_PACKED_2BIT = 0, 1
GDX_RANK_CONDENSED, GDX_RANK_FLAT = 0, 1
GDX_NCCL_UNIQUE_ID_BYTES = 128
GDX_ABI_VERSION = 2
GDX_HAMMING_MAX_MISMATCHES = 3
GDX_HAMMING_MAX_QUERY_LEN = 256


class gdx_alphabet(C.Structure):
    _fields_ = [("io_to_dense", C.c_uint8 * 256), ("num_dense_symbols", C.c_uint32),
                ("num_searchable_dense_symbols", C.c_uint32)]


class gdx_config(C.Structure):
    _fields_ = [("storage", C.c_uint32), ("suffix_array_sampling_rate", C.c_uint32),
                ("lookup_table_depth", C.c_uint32), ("performance_priority", C.c_uint32),
                ("construction", C.c_uint32), ("device", C.c_int32), ("flags", C.c_uint32),
                ("accelerator_budget_bytes", C.c_uint64)]


class gdx_hit(C.Structure):
    _fields_ = [("text_id", C.c_uint64), ("position", C.c_uint64)]


class gdx_hamming_interval(C.Structure):
    _fields_ = [("start", C.c_uint64), ("end", C.c_uint64), ("mismatches", C.c_uint32), ("reserved", C.c_uint32)]


class gdx_queries(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("offsets", C.c_void_p), ("fixed_len", C.c_uint64), ("nq", C.c_uint64),
                ("encoding", C.c_uint32), ("first_symbol", C.c_uint32)]


class gdx_parts(C.Structure):
    _fields_ = [("alphabet", gdx_alphabet), ("storage", C.c_uint32), ("text_len", C.c_uint64),
                ("count", C.c_void_p), ("interleaved_blocks", C.c_void_p),
                ("interleaved_block_offsets", C.c_void_p), ("sampled_suffix_array", C.c_void_p),
                ("sampling_rate", C.c_uint32), ("text_border_rows", C.c_void_p),
                ("text_border_positions", C.c_void_p), ("num_text_borders", C.c_uint64),
                ("sentinel_indices", C.c_void_p), ("num_texts", C.c_uint64),
                ("lookup_table_depth", C.c_uint32), ("sampled_suffix_array_u32", C.c_void_p),
                ("flags", C.c_uint32), ("accelerator_budget_bytes", C.c_uint64),
                ("rank_variant", C.c_uint32), ("block_bits", C.c_uint32)]


class gdx_index_info(C.Structure):
    _fields_ = [("text_len", C.c_uint64), ("num_texts", C.c_uint64), ("num_dense_symbols", C.c_uint32),
                ("num_searchable_dense_symbols", C.c_uint32), ("storage", C.c_uint32),
                ("sampling_rate", C.c_uint32), ("lookup_table_depth", C.c_uint32), ("rank_layout", C.c_uint32),
                ("rank_record_bytes", C.c_uint32), ("rank_positions_per_record", C.c_uint32),
                ("device", C.c_int32), ("image_bytes", C.c_uint64), ("rank_bytes", C.c_uint64),
                ("sample_bytes", C.c_uint64), ("lookup_bytes", C.c_uint64), ("num_samples", C.c_uint64),
                ("num_text_borders", C.c_uint64), ("text_bytes", C.c_uint64),
                ("inverse_sample_bytes", C.c_uint64), ("dense_suffix_array_bytes", C.c_uint64), ("seed_table_bytes", C.c_uint64),
                ("seed_table_depth", C.c_uint32), ("row_context_entry_bytes", C.c_uint32)]


class gdx_stats(C.Structure):
    _fields_ = [("queries", C.c_uint64), ("lf_steps", C.c_uint64), ("hits", C.c_uint64),
                ("walk_steps", C.c_uint64), ("kernel_ms_search", C.c_double),
                ("kernel_ms_locate", C.c_double), ("kernel_launches", C.c_uint64),
                ("verified_queries", C.c_uint64), ("locate_walk_steps", C.c_uint64),
                ("packed_queries", C.c_uint64), ("exception_queries", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("shards", C.c_uint64)]


# every symbol include/genedex_b200.h declares: name -> (restype, argtypes)
_vp, _u64, _i32, _u32 = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint32
_P = C.POINTER
PROTOTYPES = {
    "gdx_abi_version": (_u32, []),
    "gdx_last_error_message": (C.c_char_p, []),
    "gdx_last_error_query": (_u64, []),
    "gdx_device_count": (_i32, []),
    "gdx_index_build": (C.c_int, [_vp, _vp, _u64, _P(gdx_alphabet), _P(gdx_config), _P(_vp)]),
    "gdx_index_create_from_parts": (C.c_int, [_P(gdx_parts), _i32, _P(_vp)]),
    "gdx_index_create_from_bwt": (C.c_int, [_vp, _P(gdx_parts), _i32, _P(_vp)]),
    "gdx_suffix_array": (C.c_int, [_vp, _u64, _u32, _u32, _i32, _vp]),
    "gdx_concat_texts": (C.c_int, [_vp, _vp, _u64, _P(gdx_alphabet), _vp, _vp, _vp]),
    "gdx_index_download_bwt": (C.c_int, [_vp, _vp]),
    "gdx_index_get_count": (C.c_int, [_vp, _vp]),
    "gdx_index_download_samples": (C.c_int, [_vp, _vp]),
    "gdx_index_download_text_borders": (C.c_int, [_vp, _vp, _vp]),
    "gdx_index_destroy": (None, [_vp]),
    "gdx_index_get_info": (C.c_int, [_vp, _P(gdx_index_info)]),
    "gdx_index_set_dense_suffix_array": (C.c_int, [_vp, C.c_int32]),
    "gdx_index_set_seed_table_depth": (C.c_int, [_vp, C.c_int32]),
    "gdx_index_set_text_verification": (C.c_int, [_vp, C.c_int32]),
    "gdx_index_set_row_context_table": (C.c_int, [_vp, C.c_int32]),
    "gdx_index_save_to_file": (C.c_int, [_vp, C.c_char_p, _vp, _u64]),
    "gdx_index_load_from_file": (C.c_int, [C.c_char_p, _i32, _P(_vp), _vp, _u64, _P(_u64)]),
    "gdx_index_header_bytes": (_u64, []),
    "gdx_index_export": (C.c_int, [_vp, _vp, _P(_vp), _P(_u64)]),
    "gdx_index_adopt_image": (C.c_int, [_vp, _vp, _i32, _i32, _P(_vp)]),
    "gdx_index_replicate": (C.c_int, [_vp, _P(_i32), _i32, _P(_vp)]),
    "gdx_replicate_transport": (C.c_char_p, []),
    "gdx_nccl_unique_id": (C.c_int, [_vp]),
    "gdx_index_broadcast": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _P(_vp)]),
    "gdx_shard_range": (None, [_u64, _u32, _u32, _P(_u64), _P(_u64)]),
    "gdx_count_many_sharded": (C.c_int, [_P(_vp), _u32, _u32, _u32, _P(gdx_queries), _vp]),
    "gdx_cursors_many_sharded": (C.c_int, [_P(_vp), _u32, _u32, _u32, _P(gdx_queries), _vp, _vp]),
    "gdx_locate_many_sharded": (C.c_int, [_P(_vp), _u32, _u32, _u32, _P(gdx_queries), _vp, _P(_vp), _P(_u64)]),
    "gdx_count_many_u32": (C.c_int, [_vp, _P(gdx_queries), _vp]),
    "gdx_cursors_many_u32": (C.c_int, [_vp, _P(gdx_queries), _vp, _vp]),
    "gdx_packed_bytes": (_u64, [_u64]),
    "gdx_pack_queries": (C.c_int, [_vp, _P(gdx_queries), _vp, _P(_u64)]),
    "gdx_pack_symbols": (C.c_int, [_P(gdx_alphabet), _vp, _u64, _vp, _vp, _u64, _P(_u64)]),
    "gdx_cursors_many": (C.c_int, [_vp, _P(gdx_queries), _vp, _vp]),
    "gdx_count_many": (C.c_int, [_vp, _P(gdx_queries), _vp]),
    "gdx_locate_many": (C.c_int, [_vp, _P(gdx_queries), _vp, _P(_vp), _P(_u64)]),
    "gdx_locate_many_compact": (C.c_int, [_vp, _P(gdx_queries), _vp, _P(_vp), _P(_u64)]),
    "gdx_locate_many_sharded_compact": (C.c_int, [_P(_vp), _u32, _u32, _u32, _P(gdx_queries), _vp, _P(_vp), _P(_u64)]),
    "gdx_locate_intervals": (C.c_int, [_vp, _vp, _vp, _u64, _vp, _P(_vp), _P(_u64)]),
    "gdx_free_hits": (None, [_vp, _vp]),
    "gdx_extend_many": (C.c_int, [_vp, _vp, _vp, _vp, _u64]),
    "gdx_count_many_hamming": (C.c_int, [_vp, _P(gdx_queries), _u32, _vp]),
    "gdx_cursors_many_hamming": (C.c_int, [_vp, _P(gdx_queries), _u32, _vp, _P(_vp), _P(_u64)]),
    "gdx_locate_many_hamming": (C.c_int, [_vp, _P(gdx_queries), _u32, _vp, _P(_vp), _P(_u64)]),
    "gdx_cursor_for_query": (C.c_int, [_vp, _vp, _u64, _P(_u64), _P(_u64)]),
    "gdx_cursors_many_device": (C.c_int, [_vp, _P(gdx_queries), _vp, _vp, _vp, _vp]),
    "gdx_count_many_device": (C.c_int, [_vp, _P(gdx_queries), _vp, _vp, _vp]),
    "gdx_locate_intervals_device": (C.c_int, [_vp, _vp, _vp, _u64, _vp, _u64, _vp, _vp]),
    "gdx_host_pool_resize": (_u32, [_u32]),
    "gdx_host_pack_tuning": (None, [_i32, _i32]),
    "gdx_host_alloc": (C.c_int, [_u64, _P(_vp)]),
    "gdx_host_free": (None, [_vp]),
    "gdx_get_stats": (C.c_int, [_P(gdx_stats)]),
    "gdx_measure_random_gather": (C.c_int, [_i32, _u64, _u32, _u64, _i32, _P(C.c_double), _P(C.c_double)]),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"genedex_b200: {LIB_PATH} is missing. Build it with `make -C genedex_b200/csrc` "
            "(or __graft_entry__.build()); there is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError = the library does not match the header
        fn.restype = res
        fn.argtypes = args
    if lib.gdx_abi_version() != GDX_ABI_VERSION:
        raise ImportError("genedex_b200: ABI version mismatch between the Python package and the library")
    _lib = lib
    return lib
