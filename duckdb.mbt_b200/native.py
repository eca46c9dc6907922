"""ctypes binding of libduckdb_mb_gpu.so (include/duckdb_mb_gpu.h).

The product path fails loudly when the CUDA library is missing: there is no CPU fallback.
torch is used only as plumbing here (device allocations for the L0 tests / bench).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# DMB_LIB_PATH: development aid (kernel tuning variants built next to the default library)
LIB_PATH = os.environ.get("DMB_LIB_PATH") or os.path.join(_HERE, "csrc", "libduckdb_mb_gpu.so")


class VecDesc(C.Structure):
    _fields_ = [("data_off", C.c_uint64), ("val_off", C.c_int64)]


class FixedJob(C.Structure):
    _fields_ = [("in_data", C.c_void_p), ("in_validity", C.c_void_p), ("vecs", C.c_void_p),
                ("out_values", C.c_void_p), ("out_validity", C.c_void_p), ("out_valid_bytes", C.c_void_p),
                ("null_count", C.c_void_p), ("op", C.c_int32), ("param", C.c_int32)]


class StringJob(C.Structure):
    _fields_ = [("in_", C.c_void_p), ("in_validity", C.c_void_p), ("vecs", C.c_void_p),
                ("heap_dev", C.c_void_p), ("heap_host_base", C.c_uint64), ("heap_len", C.c_uint64),
                ("out_offsets", C.c_void_p), ("out_data", C.c_void_p), ("out_validity", C.c_void_p),
                ("out_valid_bytes", C.c_void_p), ("null_count", C.c_void_p), ("total_bytes", C.c_void_p),
                ("mode", C.c_int32), ("reserved", C.c_int32), ("out_data_cap", C.c_uint64)]


class RenderJob(C.Structure):
    _fields_ = [("in_data", C.c_void_p), ("in_validity", C.c_void_p), ("vecs", C.c_void_p), ("out", C.c_void_p),
                ("out_heap", C.c_void_p), ("heap_host_base", C.c_uint64), ("type_id", C.c_int32), ("phys", C.c_int32),
                ("dec_scale", C.c_int32), ("reserved", C.c_int32)]


class RevFixedJob(C.Structure):
    _fields_ = [("in_values", C.c_void_p), ("in_validity", C.c_void_p), ("in_bit_offset", C.c_int64),
                ("out_data", C.c_void_p), ("out_validity", C.c_void_p), ("null_count", C.c_void_p),
                ("op", C.c_int32), ("reserved", C.c_int32)]


class RevStringJob(C.Structure):
    _fields_ = [("in_offsets", C.c_void_p), ("in_data", C.c_void_p), ("in_validity", C.c_void_p),
                ("in_bit_offset", C.c_int64), ("data_host_base", C.c_uint64), ("out", C.c_void_p),
                ("out_validity", C.c_void_p), ("null_count", C.c_void_p), ("large_offsets", C.c_int32),
                ("reserved", C.c_int32)]


class RevListJob(C.Structure):
    _fields_ = [("in_offsets", C.c_void_p), ("in_validity", C.c_void_p), ("in_bit_offset", C.c_int64),
                ("in_child_validity", C.c_void_p), ("child_bit_offset", C.c_int64), ("child_word", C.c_void_p),
                ("out_entries", C.c_void_p), ("out_validity", C.c_void_p), ("out_child_validity", C.c_void_p),
                ("null_count", C.c_void_p), ("error", C.c_void_p), ("large_offsets", C.c_int32), ("reserved", C.c_int32)]


class EnumDict(C.Structure):
    _fields_ = [("size", C.c_uint32), ("reserved", C.c_uint32), ("offsets", C.c_void_p), ("data", C.c_void_p)]


class EnumJob(C.Structure):
    _fields_ = [("in_data", C.c_void_p), ("in_validity", C.c_void_p), ("vecs", C.c_void_p), ("out", C.c_void_p),
                ("dict_offsets", C.c_void_p), ("dict_data", C.c_void_p), ("dict_host_base", C.c_uint64),
                ("bad_index", C.c_void_p), ("dict_size", C.c_uint32), ("phys", C.c_int32)]


class ListJob(C.Structure):
    _fields_ = [("in_entries", C.c_void_p), ("in_validity", C.c_void_p), ("vecs", C.c_void_p), ("child_base", C.c_void_p),
                ("child_data", C.c_void_p), ("child_validity", C.c_void_p), ("child_val_off", C.c_void_p),
                ("out_offsets", C.c_void_p), ("out_child", C.c_void_p), ("out_child_validity", C.c_void_p),
                ("total", C.c_void_p), ("child_null_count", C.c_void_p), ("child_width", C.c_int32), ("large", C.c_int32),
                ("child_sizes", C.c_void_p)]


class HostColumn(C.Structure):
    pass


class HostList(C.Structure):
    _fields_ = [("child_type_id", C.c_int32), ("child_phys", C.c_int32), ("child_dec_width", C.c_int32), ("child_dec_scale", C.c_int32),
                ("child_data", C.c_void_p), ("child_validity", C.c_void_p), ("child_sizes", C.c_void_p),
                ("child_col", C.POINTER(HostColumn))]


class HostStruct(C.Structure):
    _fields_ = [("nfields", C.c_int32), ("reserved", C.c_int32), ("fields", C.POINTER(HostColumn))]


HostColumn._fields_ = [("name", C.c_char_p), ("type_id", C.c_int32), ("phys", C.c_int32), ("dec_width", C.c_int32),
                       ("dec_scale", C.c_int32), ("data", C.POINTER(C.c_void_p)), ("validity", C.POINTER(C.c_void_p)),
                       ("heap_base", C.c_void_p), ("heap_len", C.c_uint64), ("dict", C.POINTER(EnumDict)), ("list", C.POINTER(HostList)),
                       ("struct_", C.POINTER(HostStruct))]


class HostBatch(C.Structure):
    _fields_ = [("ncols", C.c_int32), ("flags", C.c_int32), ("nchunks", C.c_int64), ("counts", C.c_void_p),
                ("cols", C.POINTER(HostColumn))]


class ArrowSchema(C.Structure):
    pass


ArrowSchema._fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_char_p), ("flags", C.c_int64),
                        ("n_children", C.c_int64), ("children", C.POINTER(C.POINTER(ArrowSchema))),
                        ("dictionary", C.POINTER(ArrowSchema)), ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowArray(C.Structure):
    pass


ArrowArray._fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
                       ("n_children", C.c_int64), ("buffers", C.POINTER(C.c_void_p)),
                       ("children", C.POINTER(C.POINTER(ArrowArray))), ("dictionary", C.POINTER(ArrowArray)),
                       ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowArrayStream(C.Structure):  # Arrow C stream interface: 5 pointers
    _fields_ = [("get_schema", C.c_void_p), ("get_next", C.c_void_p), ("get_last_error", C.c_void_p), ("release", C.c_void_p),
                ("private_data", C.c_void_p)]


class TypedColumn(C.Structure):
    _fields_ = [("tag", C.c_int32), ("width", C.c_int32), ("length", C.c_int64), ("null_count", C.c_int64),
                ("values", C.c_void_p), ("valid", C.c_void_p), ("offsets", C.c_void_p), ("data", C.c_void_p)]


CHUNK_SINK = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_int32, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p))

# every symbol include/duckdb_mb_gpu.h declares (checked by tests/test_abi.py without a GPU)
EXPORTED_SYMBOLS = [
    "dmb_dev_fixed_batch", "dmb_op_out_width", "dmb_phys_width", "dmb_dev_string_scratch_bytes",
    "dmb_dev_string_error", "dmb_dev_string_batch", "dmb_dev_set_lookback_limit_ns", "dmb_dev_rev_fixed_batch", "dmb_dev_rev_string_batch",
    "dmb_dev_rev_list_batch", "dmb_rev_list_cut",
    "dmb_dev_valid_bytes_to_masks", "dmb_dev_make_string_t", "dmb_dev_blob_escape", "dmb_render_supported", "dmb_render_slot_bytes", "dmb_dev_render_text", "dmb_dev_enum_to_string_t", "dmb_dev_enum_utf8", "dmb_dev_list_scratch_bytes", "dmb_dev_list_batch",
    "duckdb_mb_gpu_last_error", "duckdb_mb_gpu_device_count", "duckdb_mb_gpu_bind_numa", "duckdb_mb_gpu_ctx_create",
    "duckdb_mb_gpu_ctx_destroy", "duckdb_mb_gpu_ctx_sync", "duckdb_mb_gpu_host_alloc", "duckdb_mb_gpu_host_free",
    "duckdb_mb_gpu_result_from_chunks", "duckdb_mb_gpu_result_materialise_arrow",
    "duckdb_mb_gpu_result_export_arrow", "duckdb_mb_gpu_result_typed_column", "duckdb_mb_gpu_result_text_column", "duckdb_mb_gpu_result_timings",
    "duckdb_mb_gpu_result_link_bytes",
    "duckdb_mb_arrow_column_count", "duckdb_mb_arrow_row_count", "duckdb_mb_arrow_schema",
    "duckdb_mb_arrow_get_column_int32", "duckdb_mb_arrow_get_column_int64", "duckdb_mb_arrow_get_column_double",
    "duckdb_mb_arrow_get_column_string", "duckdb_mb_arrow_get_column_bool",
    "duckdb_mb_arrow_get_column_int32_nullable", "duckdb_mb_arrow_get_column_int64_nullable",
    "duckdb_mb_arrow_get_column_double_nullable", "duckdb_mb_arrow_get_column_string_nullable",
    "duckdb_mb_arrow_get_column_bool_nullable", "duckdb_mb_arrow_destroy", "duckdb_mb_is_null_arrow_result",
    "duckdb_mb_result_destroy", "duckdb_mb_is_null_result", "duckdb_mb_result_column_count", "duckdb_mb_result_row_count",
    "duckdb_mb_result_column_name", "duckdb_mb_result_column_type", "duckdb_mb_result_is_null", "duckdb_mb_result_value",
    "duckdb_mb_gpu_stream_from_result", "duckdb_mb_stream_destroy", "duckdb_mb_is_null_stream", "duckdb_mb_stream_column_count",
    "duckdb_mb_stream_column_name", "duckdb_mb_stream_fetch_chunk", "duckdb_mb_chunk_destroy", "duckdb_mb_is_null_chunk",
    "duckdb_mb_chunk_row_count", "duckdb_mb_chunk_column_count", "duckdb_mb_chunk_is_null", "duckdb_mb_chunk_value",
    "duckdb_mb_bytes_to_double",
    "duckdb_mb_gpu_result_set_owner", "duckdb_mb_gpu_stream_from_result_owned", "duckdb_mb_gpu_appender_set_hooks",
    "duckdb_mb_gpu_result_from_chunks_sharded", "duckdb_mb_gpu_result_shard", "duckdb_mb_gpu_sharded_part_count", "duckdb_mb_gpu_sharded_part",
    "duckdb_mb_gpu_sharded_first_row", "duckdb_mb_gpu_sharded_materialise_arrow", "duckdb_mb_gpu_sharded_string_bases",
    "duckdb_mb_gpu_sharded_destroy", "duckdb_mb_gpu_sharded_export_stream", "duckdb_mb_gpu_result_export_stream",
    # the reference's appender symbols (src/duckdb_native.c:1083-1251, 1313-1533, 1735-1926)
    "duckdb_mb_appender_destroy", "duckdb_mb_appender_error", "duckdb_mb_is_null_appender", "duckdb_mb_begin_row",
    "duckdb_mb_append_int", "duckdb_mb_append_bigint", "duckdb_mb_append_double", "duckdb_mb_append_varchar", "duckdb_mb_append_bool",
    "duckdb_mb_append_null", "duckdb_mb_end_row", "duckdb_mb_flush", "duckdb_mb_append_date", "duckdb_mb_append_timestamp",
    "duckdb_mb_append_blob", "duckdb_mb_append_decimal", "duckdb_mb_append_interval", "duckdb_mb_append_list_varchar",
    "duckdb_mb_append_struct_varchar", "duckdb_mb_append_map_varchar_varchar",
    "duckdb_mb_gpu_appender_create", "duckdb_mb_gpu_appender_destroy", "duckdb_mb_gpu_appender_error",
    "duckdb_mb_gpu_appender_state", "duckdb_mb_gpu_appender_row_count", "duckdb_mb_gpu_append_arrow_batch",
    "duckdb_mb_gpu_appender_flush", "duckdb_mb_gpu_appender_close", "duckdb_mb_gpu_appender_timings",
    "duckdb_mb_gpu_appender_flushed_row_count", "duckdb_mb_gpu_appender_link_bytes",
    "duckdb_mb_gpu_begin_row", "duckdb_mb_gpu_append_int", "duckdb_mb_gpu_append_bigint", "duckdb_mb_gpu_append_double",
    "duckdb_mb_gpu_append_varchar", "duckdb_mb_gpu_append_bool", "duckdb_mb_gpu_append_null", "duckdb_mb_gpu_append_date",
    "duckdb_mb_gpu_append_timestamp", "duckdb_mb_gpu_end_row", "duckdb_mb_gpu_append_blob", "duckdb_mb_gpu_append_decimal",
    "duckdb_mb_gpu_append_list_varchar", "duckdb_mb_gpu_append_struct_varchar", "duckdb_mb_gpu_append_map_varchar_varchar",
    "duckdb_mb_gpu_append_interval", "duckdb_mb_gpu_appender_set_decimal", "duckdb_mb_gpu_appender_set_list",
    "duckdb_mb_gpu_appender_list_child",
]

_lib = None


class NativeLibraryMissing(RuntimeError):
    pass


def lib():
    """Load the CUDA library.  No fallback: a missing build is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryMissing(
            f"{LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the product path)")
    L = C.CDLL(LIB_PATH)
    missing = [s for s in EXPORTED_SYMBOLS if not hasattr(L, s)]
    if missing and not os.environ.get("DMB_ALLOW_PARTIAL"):
        raise NativeLibraryMissing(f"{LIB_PATH} is stale or partial, missing symbols: {missing}; rebuild it")
    real = L

    class _Partial:  # development aid only (DMB_ALLOW_PARTIAL=1): signatures of absent symbols are ignored
        def __getattr__(self, name):
            if hasattr(real, name):
                return getattr(real, name)
            return type("_Absent", (), {})()

    L = _Partial() if missing else real
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.duckdb_mb_gpu_last_error.restype = C.c_char_p
    L.dmb_dev_fixed_batch.restype = i32
    L.dmb_dev_fixed_batch.argtypes = [vp, vp, i32, vp, vp, i64, i64, vp]
    L.dmb_op_out_width.restype = i32
    L.dmb_op_out_width.argtypes = [i32]
    L.dmb_phys_width.restype = i32
    L.dmb_phys_width.argtypes = [i32]
    L.dmb_dev_string_scratch_bytes.restype = C.c_size_t
    L.dmb_dev_string_scratch_bytes.argtypes = [i64]
    L.dmb_dev_string_batch.restype = i32
    L.dmb_dev_string_batch.argtypes = [C.POINTER(StringJob), vp, vp, i64, i64, vp, vp]
    L.dmb_dev_string_error.restype = i32
    L.dmb_dev_string_error.argtypes = [vp, vp]
    L.dmb_dev_make_string_t.restype = i32
    L.dmb_dev_make_string_t.argtypes = [vp, vp, vp, u64, vp, i64, vp]
    L.dmb_render_supported.restype = i32
    L.dmb_render_supported.argtypes = [i32, i32]
    L.dmb_dev_render_text.restype = i32
    L.dmb_dev_render_text.argtypes = [C.POINTER(RenderJob), vp, i64, vp]
    L.dmb_dev_valid_bytes_to_masks.restype = i32
    L.dmb_dev_valid_bytes_to_masks.argtypes = [vp, vp, vp, i64, vp]
    L.dmb_dev_enum_to_string_t.restype = i32
    L.dmb_dev_enum_to_string_t.argtypes = [C.POINTER(EnumJob), vp, i64, vp]
    L.dmb_dev_enum_utf8.restype = i32
    L.dmb_dev_enum_utf8.argtypes = [C.POINTER(EnumJob), C.POINTER(StringJob), vp, vp, i64, i64, vp, vp]
    L.dmb_dev_list_scratch_bytes.restype = C.c_size_t
    L.dmb_dev_list_scratch_bytes.argtypes = [i64]
    L.dmb_dev_list_batch.restype = i32
    L.dmb_dev_list_batch.argtypes = [C.POINTER(ListJob), vp, vp, i64, i64, i64, vp, vp]
    L.dmb_dev_rev_fixed_batch.restype = i32
    L.dmb_dev_rev_fixed_batch.argtypes = [vp, vp, i32, i64, vp]
    L.dmb_dev_rev_string_batch.restype = i32
    L.dmb_dev_rev_string_batch.argtypes = [C.POINTER(RevStringJob), i64, vp]
    L.dmb_dev_rev_list_batch.restype = i32
    L.dmb_dev_rev_list_batch.argtypes = [C.POINTER(RevListJob), i64, vp]
    L.dmb_rev_list_cut.restype = i64
    L.dmb_rev_list_cut.argtypes = [vp, i32, i64, i64, i64, i64]
    L.duckdb_mb_gpu_appender_list_child.restype = i32
    L.duckdb_mb_gpu_appender_list_child.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]
    L.duckdb_mb_gpu_device_count.restype = i32
    L.duckdb_mb_gpu_ctx_create.restype = vp
    L.duckdb_mb_gpu_ctx_create.argtypes = [i32]
    L.duckdb_mb_gpu_ctx_destroy.argtypes = [vp]
    L.duckdb_mb_gpu_ctx_sync.restype = i32
    L.duckdb_mb_gpu_ctx_sync.argtypes = [vp]
    L.duckdb_mb_gpu_host_alloc.restype = vp
    L.duckdb_mb_gpu_host_alloc.argtypes = [C.c_size_t]
    L.duckdb_mb_gpu_host_free.argtypes = [vp]
    L.duckdb_mb_gpu_result_from_chunks.restype = vp
    L.duckdb_mb_gpu_result_from_chunks.argtypes = [vp, C.POINTER(HostBatch)]
    L.duckdb_mb_gpu_result_materialise_arrow.restype = i32
    L.duckdb_mb_gpu_result_materialise_arrow.argtypes = [vp]
    L.duckdb_mb_gpu_result_export_arrow.restype = i32
    L.duckdb_mb_gpu_result_export_arrow.argtypes = [vp, i32, vp, vp]
    L.duckdb_mb_gpu_result_from_chunks_sharded.restype = vp
    L.duckdb_mb_gpu_result_from_chunks_sharded.argtypes = [C.POINTER(vp), i32, vp]
    L.duckdb_mb_gpu_result_shard.restype = vp
    L.duckdb_mb_gpu_result_shard.argtypes = [vp, C.POINTER(vp), i32, i64]
    L.duckdb_mb_gpu_sharded_part_count.argtypes = [vp]
    L.duckdb_mb_gpu_sharded_part.restype = vp
    L.duckdb_mb_gpu_sharded_part.argtypes = [vp, i32]
    L.duckdb_mb_gpu_sharded_first_row.restype = i64
    L.duckdb_mb_gpu_sharded_first_row.argtypes = [vp, i32]
    L.duckdb_mb_gpu_sharded_materialise_arrow.argtypes = [vp]
    L.duckdb_mb_gpu_sharded_string_bases.argtypes = [vp, i32, vp]
    L.duckdb_mb_gpu_sharded_destroy.argtypes = [vp]
    L.duckdb_mb_gpu_sharded_export_stream.argtypes = [vp, vp]
    L.duckdb_mb_gpu_result_export_stream.argtypes = [vp, i64, vp]
    L.duckdb_mb_gpu_result_typed_column.restype = i32
    L.duckdb_mb_gpu_result_typed_column.argtypes = [vp, i32, C.POINTER(TypedColumn)]
    L.duckdb_mb_gpu_result_text_column.restype = i32
    L.duckdb_mb_gpu_result_text_column.argtypes = [vp, i32, C.POINTER(TypedColumn)]
    L.duckdb_mb_gpu_result_timings.restype = i32
    L.duckdb_mb_gpu_result_timings.argtypes = [vp, C.POINTER(C.c_double)]
    L.duckdb_mb_gpu_result_link_bytes.restype = i32
    L.duckdb_mb_gpu_result_link_bytes.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.duckdb_mb_arrow_column_count.restype = i32
    L.duckdb_mb_arrow_column_count.argtypes = [vp]
    L.duckdb_mb_arrow_row_count.restype = i32
    L.duckdb_mb_arrow_row_count.argtypes = [vp]
    L.duckdb_mb_arrow_schema.restype = vp
    L.duckdb_mb_arrow_schema.argtypes = [vp]
    for kind in ("int32", "int64", "double", "string", "bool"):
        for suffix in ("", "_nullable"):
            f = getattr(L, f"duckdb_mb_arrow_get_column_{kind}{suffix}")
            f.restype = vp
            f.argtypes = [vp, i32]
    L.duckdb_mb_arrow_destroy.argtypes = [vp]
    L.duckdb_mb_is_null_arrow_result.restype = i32
    L.duckdb_mb_is_null_arrow_result.argtypes = [vp]
    # per-cell drop-ins (materialised result, streaming chunks)
    for name in ("duckdb_mb_result_destroy", "duckdb_mb_stream_destroy", "duckdb_mb_chunk_destroy"):
        getattr(L, name).restype = None
        getattr(L, name).argtypes = [vp]
    for name in ("duckdb_mb_is_null_result", "duckdb_mb_result_column_count", "duckdb_mb_result_row_count", "duckdb_mb_is_null_stream",
                 "duckdb_mb_stream_column_count", "duckdb_mb_is_null_chunk", "duckdb_mb_chunk_row_count", "duckdb_mb_chunk_column_count"):
        getattr(L, name).restype = i32
        getattr(L, name).argtypes = [vp]
    for name in ("duckdb_mb_result_column_name", "duckdb_mb_stream_column_name"):
        getattr(L, name).restype = vp
        getattr(L, name).argtypes = [vp, i32]
    L.duckdb_mb_result_column_type.restype = i32
    L.duckdb_mb_result_column_type.argtypes = [vp, i32]
    for name in ("duckdb_mb_result_is_null", "duckdb_mb_chunk_is_null"):
        getattr(L, name).restype = i32
        getattr(L, name).argtypes = [vp, i32, i32]
    for name in ("duckdb_mb_result_value", "duckdb_mb_chunk_value"):
        getattr(L, name).restype = vp
        getattr(L, name).argtypes = [vp, i32, i32]
    L.duckdb_mb_gpu_stream_from_result.restype = vp
    L.duckdb_mb_gpu_stream_from_result.argtypes = [vp]
    L.duckdb_mb_stream_fetch_chunk.restype = vp
    L.duckdb_mb_stream_fetch_chunk.argtypes = [vp]
    L.duckdb_mb_bytes_to_double.restype = C.c_double
    L.duckdb_mb_bytes_to_double.argtypes = [vp, i32]
    L.duckdb_mb_gpu_appender_create.restype = vp
    L.duckdb_mb_gpu_appender_create.argtypes = [vp, i32, vp, CHUNK_SINK, vp]
    L.duckdb_mb_gpu_appender_destroy.argtypes = [vp]
    L.duckdb_mb_gpu_appender_error.restype = vp
    L.duckdb_mb_gpu_appender_error.argtypes = [vp]
    L.duckdb_mb_gpu_appender_state.restype = i32
    L.duckdb_mb_gpu_appender_state.argtypes = [vp]
    L.duckdb_mb_gpu_appender_row_count.restype = i64
    L.duckdb_mb_gpu_appender_row_count.argtypes = [vp]
    L.duckdb_mb_gpu_append_arrow_batch.restype = i32
    L.duckdb_mb_gpu_append_arrow_batch.argtypes = [vp, vp, vp]
    L.duckdb_mb_gpu_appender_flush.restype = i32
    L.duckdb_mb_gpu_appender_flush.argtypes = [vp]
    L.duckdb_mb_gpu_appender_close.restype = i32
    L.duckdb_mb_gpu_appender_close.argtypes = [vp]
    L.duckdb_mb_gpu_appender_timings.restype = i32
    L.duckdb_mb_gpu_appender_timings.argtypes = [vp, C.POINTER(C.c_double)]
    L.duckdb_mb_gpu_appender_flushed_row_count.restype = i64
    L.duckdb_mb_gpu_appender_flushed_row_count.argtypes = [vp]
    L.duckdb_mb_gpu_appender_link_bytes.restype = i32
    L.duckdb_mb_gpu_appender_link_bytes.argtypes = [vp, C.POINTER(C.c_uint64)]
    for name, extra in (("begin_row", []), ("append_int", [i32]), ("append_bigint", [i64]), ("append_double", [C.c_double]),
                        ("append_varchar", [C.c_char_p, i32]), ("append_bool", [i32]), ("append_null", []),
                        ("append_date", [i32]), ("append_timestamp", [i64]), ("end_row", []),
                        ("append_blob", [C.c_char_p, i32]), ("append_decimal", [i32, i32, i64, i64]),
                        ("append_interval", [i32, i32, i64]), ("appender_set_decimal", [i32, i32, i32]),
                        ("appender_set_list", [i32, i32, i32, i32]),
                        ("append_list_varchar", [vp, vp, i32]), ("append_struct_varchar", [vp, vp, vp, vp, i32]),
                        ("append_map_varchar_varchar", [vp, vp, vp, vp, i32])):
        f = getattr(L, "duckdb_mb_gpu_" + name)
        f.restype = i32
        f.argtypes = [vp] + extra
    _lib = real
    return real


def last_error() -> str:
    return (lib().duckdb_mb_gpu_last_error() or b"").decode(errors="replace")


def check(rc: int, what: str) -> None:
    if rc < 0:
        raise RuntimeError(f"{what}: {last_error()}")


class MoonbitBlob:
    """A moonbit_bytes_t viewed in place (no copy) as a numpy uint8 array; freed on exit.  The decoder mirror reads the
    blob exactly once, like the MoonBit decoders do."""

    def __init__(self, ptr: Optional[int]):
        self.ptr = ptr
        self.view = np.zeros(0, dtype=np.uint8)
        if ptr:
            n = C.c_uint32.from_address(ptr - 4).value
            if n:
                self.view = np.ctypeslib.as_array((C.c_uint8 * n).from_address(ptr))

    def __enter__(self):
        return self.view

    def __exit__(self, *exc):
        self.view = None
        if self.ptr:
            C.CDLL(None).free(C.c_void_p(self.ptr - 8))
            self.ptr = None


def moonbit_bytes(ptr: Optional[int]) -> bytes:
    """Copy a moonbit_bytes_t out (stand-in header: [int32 rc][uint32 len] before the payload,
    include/moonbit_standin.h) and free it."""
    if not ptr:
        return b""
    n = C.c_uint32.from_address(ptr - 4).value
    data = C.string_at(ptr, n)
    C.CDLL(None).free(C.c_void_p(ptr - 8))
    return data
