"""ctypes binding of libcsvb200.so -- exactly the symbols include/csvb200.h declares.

The library is built in-tree by csv_simd_b200/build.py (nvcc, sm_100a).  If it is missing and
cannot be built this module raises: there is no CPU fallback anywhere in the product path.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
szp = C.POINTER(C.c_size_t)
vpp = C.POINTER(C.c_void_p)


class Range(C.Structure):
    _fields_ = [("start", C.c_uint64), ("end", C.c_uint64)]


class StreamStats(C.Structure):
    _fields_ = [("bytes", C.c_uint64), ("entries", C.c_uint64), ("seconds", C.c_double), ("chunks", C.c_uint32),
                ("end_parity", C.c_int)]


READ_FN = C.CFUNCTYPE(C.c_size_t, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)
SINK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.c_size_t, C.c_uint64)


class TapeReport(C.Structure):
    _fields_ = [("index_len", C.c_uint64), ("jump", C.c_uint64), ("problem", C.c_uint64),
                ("first_bad_slot", C.c_uint64), ("first_bad_record", C.c_uint64), ("first_bad_pos", C.c_uint64),
                ("record_cnt", C.c_uint32), ("ok", C.c_uint32)]


class ShardInfo(C.Structure):
    _fields_ = [("base", C.c_uint64), ("entries", C.c_uint64), ("epoch", C.c_uint64), ("carry_in", C.c_uint32),
                ("redone", C.c_uint32), ("rank", C.c_uint32), ("world", C.c_uint32)]


class MultiStats(C.Structure):
    _fields_ = [("seconds", C.c_double), ("upload_seconds", C.c_double), ("download_seconds", C.c_double),
                ("entries", C.c_uint64), ("redone_mask", C.c_uint32), ("carry_mask", C.c_uint32)]


class Chunk(C.Structure):
    _fields_ = [("start", C.c_uint64), ("end", C.c_uint64), ("byte_start", C.c_uint64), ("byte_end", C.c_uint64),
                ("record_cnt", C.c_uint32), ("id", C.c_uint8)]


# name -> (restype, argtypes); kept in sync with include/csvb200.h (tests/test_abi.py checks it)
SIGNATURES = {
    "csvb200_version": (C.c_int, []),
    "csvb200_status_string": (C.c_char_p, [C.c_int]),
    "csvb200_ctx_create": (C.c_int, [C.c_int, vpp]),
    "csvb200_ctx_destroy": (None, [C.c_void_p]),
    "csvb200_last_error": (C.c_char_p, [C.c_void_p]),
    "csvb200_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "csvb200_ctx_set_reserve": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "csvb200_ctx_last_build_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "csvb200_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "csvb200_host_alloc": (C.c_int, [C.c_size_t, vpp]),
    "csvb200_host_free": (C.c_int, [C.c_void_p]),
    "csvb200_host_register": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int]),
    "csvb200_host_unregister": (C.c_int, [C.c_void_p]),
    "csvb200_index_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, vpp]),
    "csvb200_index_build_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, vpp]),
    "csvb200_index_build_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, szp]),
    "csvb200_index_build_stream": (C.c_int, [C.c_void_p, READ_FN, C.c_void_p, SINK_FN, C.c_void_p, C.c_size_t,
                                             C.POINTER(StreamStats)]),
    "csvb200_index_build_file": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, szp,
                                           C.POINTER(StreamStats)]),
    "csvb200_shard_quote_parity": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, u32p]),
    "csvb200_index_build_shard_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64,
                                                   C.c_int, vpp]),
    "csvb200_shard_quote_parity_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_index_build_shard_device_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32,
                                                      C.c_uint64, C.c_int, C.c_void_p, vpp]),
    "csvb200_index_build_shard_speculative": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64,
                                                        C.c_int, C.c_uint64, C.c_void_p, vpp]),
    "csvb200_index_shard_verify": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "csvb200_index_shard_redone": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "csvb200_shard_build_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64, C.c_int,
                                              C.c_void_p, C.c_size_t, szp, C.c_void_p, vpp]),
    "csvb200_shard_job_verify": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, szp, C.POINTER(C.c_int)]),
    "csvb200_shard_job_free": (None, [C.c_void_p]),
    "csvb200_exchange_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, vpp]),
    "csvb200_exchange_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "csvb200_exchange_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "csvb200_exchange_connect_local": (C.c_int, [vpp, C.c_uint32]),
    "csvb200_exchange_destroy": (None, [C.c_void_p]),
    "csvb200_index_build_shard_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64,
                                                     C.c_uint64, vpp]),
    "csvb200_index_shard_info": (C.c_int, [C.c_void_p, C.POINTER(ShardInfo)]),
    "csvb200_exchange_counts": (C.c_int, [C.c_void_p, C.c_void_p, u64p, u32p]),
    "csvb200_shard_build_to_host_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64,
                                                       C.c_void_p, C.c_size_t, szp, C.POINTER(ShardInfo), u64p, u32p]),
    "csvb200_multi_create": (C.c_int, [C.POINTER(C.c_int), C.c_int, vpp]),
    "csvb200_multi_destroy": (None, [C.c_void_p]),
    "csvb200_multi_last_error": (C.c_char_p, [C.c_void_p]),
    "csvb200_multi_device_count": (C.c_int, [C.c_void_p]),
    "csvb200_multi_index_build_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, szp, C.c_void_p, C.c_size_t,
                                                    szp]),
    "csvb200_multi_last_stats": (C.c_int, [C.c_void_p, C.POINTER(MultiStats)]),
    "csvb200_multi_index_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, szp, vpp]),
    "csvb200_multi_index_free": (None, [C.c_void_p]),
    "csvb200_multi_index_len": (C.c_size_t, [C.c_void_p]),
    "csvb200_multi_index_segment": (C.c_int, [C.c_void_p, C.c_int, u64p, u64p, C.POINTER(C.c_int)]),
    "csvb200_multi_index_copy_out": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "csvb200_multi_tape_init": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, u32p, u64p]),
    "csvb200_multi_seek_fields": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_multi_seek_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_multi_seek_fields_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_multi_stream": (C.c_void_p, [C.c_void_p, C.c_int]),
    "csvb200_multi_materialize_columns": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                                    vpp, vpp, szp, szp]),
    "csvb200_multi_tape_validate": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.POINTER(TapeReport)]),
    "csvb200_multi_validate_utf8": (C.c_int, [C.c_void_p, u64p, C.POINTER(C.c_int)]),
    "csvb200_multi_tape_chunks": (C.c_int, [C.c_void_p, C.c_uint8, C.POINTER(Chunk), C.c_size_t, szp]),
    "csvb200_index_wrap_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, vpp]),
    "csvb200_index_sync": (C.c_int, [C.c_void_p]),
    "csvb200_index_len": (C.c_size_t, [C.c_void_p]),
    "csvb200_index_end_parity": (C.c_int, [C.c_void_p]),
    "csvb200_index_device_ptr": (C.c_void_p, [C.c_void_p]),
    "csvb200_index_copy_out": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "csvb200_index_free": (None, [C.c_void_p]),
    "csvb200_tape_init": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, u32p, u64p]),
    "csvb200_tape_validate": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.POINTER(TapeReport)]),
    "csvb200_tape_chunks": (C.c_int, [C.c_void_p, C.c_uint8, C.POINTER(Chunk), C.c_size_t, szp]),
    "csvb200_seek_record": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(Range), C.POINTER(C.c_int)]),
    "csvb200_seek_field": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(Range), C.POINTER(C.c_int)]),
    "csvb200_seek_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_seek_fields": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_seek_fields_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_seek_records_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_gather_fields": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.c_size_t]),
    "csvb200_seek_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_void_p,
                                      C.c_size_t, szp, C.c_void_p]),
    "csvb200_seek_values_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_multi_seek_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                            C.c_void_p, C.c_size_t, szp, C.c_void_p]),
    "csvb200_multi_seek_values_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32,
                                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_materialize_column": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                             C.c_void_p, C.c_size_t, szp]),
    "csvb200_materialize_column_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                                    C.c_void_p, C.c_void_p, C.c_size_t]),
    "csvb200_materialize_columns": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                              vpp, vpp, szp, szp]),
    "csvb200_materialize_columns_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                                     vpp, vpp, szp]),
    "csvb200_validate_utf8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, u64p, C.POINTER(C.c_int)]),
    "csvb200_validate_utf8_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "csvb200_index_validation": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), u64p]),
    "csvb200_index_validate_utf8": (C.c_int, [C.c_void_p, u64p]),
    "csvb200_index_save": (C.c_int, [C.c_void_p, C.c_char_p]),
    "csvb200_index_load": (C.c_int, [C.c_void_p, C.c_char_p, vpp]),
    "csvb200_block_masks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "csvb200_class_bytes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}

_lib = None


def so_path() -> str:
    return _build.SO


def load():
    """Load (building first if stale and nvcc exists) and type the library. Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.is_stale():
        _build.build()
    if not os.path.exists(_build.SO):
        raise RuntimeError("libcsvb200.so is missing and could not be built; there is no CPU fallback")
    lib = C.CDLL(_build.SO)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header / library drift: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
