"""Host-side mirror of the reference's `Appender` (src/duckdb_native.mbt:955-1076) over the GPU
reverse path, with the protocol of src/duckdb_appender_state_machine.mbt:54-239.

Same method names and failure convention as the reference (`begin_row`, `append_int`,
`append_bigint`, `append_double`, `append_varchar`, `append_bool`, `append_null`, `end_row`,
`flush`, `close`: a failing call raises `DuckDBError` carrying the per-handle error string, where
the reference returns `Err(DuckDBError::Message(appender_error(..)))`), plus the additive bulk
door `append_arrow(record_batch)`.

Finished 2048-row chunks are handed to `sink(count, vec_data, vec_validity)`: host pointers laid
out as duckdb_vector_get_data / duckdb_vector_get_validity expect, i.e. what the glue passes to
duckdb_append_data_chunk (src/duckdb_native.c:2109-2132).  libduckdb is not in this image, so the
default sink collects the chunks (`CollectedChunks`) for inspection.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence

import numpy as np

from . import chunks as ch
from . import native as nat
from .arrow_result import DuckDBError, GpuContext

NOT_CREATED, READY, ROW_IN_PROGRESS, FLUSHED, CLOSED, ERROR = range(6)  # AppenderState, :7-14
STATE_NAMES = ["NotCreated", "Ready", "RowInProgress", "Flushed", "Closed", "Error"]


def _out_width(type_id: int, dec_width: int = 0) -> int:
    if type_id == ch.T_LIST:
        return 16  # duckdb_list_entry {uint64 offset, uint64 length}
    return ch.PHYS_WIDTH[ch.phys_of_type(type_id, dec_width)]


# numpy dtype of a fixed-width LIST child value, by physical type (128-bit ones are decoded by hand)
_CHILD_DTYPE = {ch.P_BOOL: np.uint8, ch.P_I8: np.int8, ch.P_I16: np.int16, ch.P_I32: np.int32, ch.P_I64: np.int64,
                ch.P_U8: np.uint8, ch.P_U16: np.uint16, ch.P_U32: np.uint32, ch.P_U64: np.uint64,
                ch.P_F32: np.float32, ch.P_F64: np.float64}


class CollectedChunks:
    """Default sink: copies every chunk out of the appender's pinned buffers.

    `dec_widths`: per column, the table's DECIMAL width (what `Appender.set_decimal` declares), which sets the vector's
    physical width; the Arrow precision does not.  `list_children` maps a LIST column to its child type, `(child_type_id, child_dec_width)`; for those columns the
    chunk's child vector is copied too (through Appender.list_child, valid only inside the sink call)."""

    def __init__(self, type_ids: Sequence[int], dec_widths: Optional[Sequence[int]] = None, list_children: Optional[dict] = None):
        self.type_ids = list(type_ids)
        self.widths = [_out_width(t, (dec_widths or [0] * len(type_ids))[i]) for i, t in enumerate(type_ids)]
        self.counts: List[int] = []
        self.data: List[List[bytes]] = [[] for _ in type_ids]
        self.validity: List[List[np.ndarray]] = [[] for _ in type_ids]
        self.list_children = dict(list_children or {})
        self.child_data: dict = {c: [] for c in self.list_children}      # per chunk: child values, raw bytes
        self.child_validity: dict = {c: [] for c in self.list_children}  # per chunk: ceil(size / 64) mask words
        self.appender: Optional["Appender"] = None  # set by the Appender this sink is given to

    def __call__(self, count: int, vec_data, vec_validity) -> bool:
        self.counts.append(count)
        for c, w in enumerate(self.widths):
            self.data[c].append(C.string_at(vec_data[c], count * w))
            self.validity[c].append(np.frombuffer(C.string_at(vec_validity[c], 8 * ch.VALIDITY_WORDS), dtype=np.uint64).copy())
        for c, (ct, dw) in self.list_children.items():
            data, words, size = self.appender.list_child(c)
            self.child_data[c].append(C.string_at(data, size * _out_width(ct, dw)) if size else b"")
            nw = (size + 63) // 64
            self.child_validity[c].append(np.frombuffer(C.string_at(words, 8 * nw), dtype=np.uint64).copy() if nw else np.zeros(0, np.uint64))
        return True

    def list_values(self, c: int) -> list:
        """LIST column `c` as Python lists (None: a NULL row or element).  Values: int (integers, DATE days,
        TIME / TIMESTAMP ticks, DECIMAL unscaled, HUGEINT / UHUGEINT / UUID as 128-bit integers), float, bool, str
        (VARCHAR) or bytes (BLOB).  Pointer string_t refer to the Arrow data buffer, which must still be alive."""
        ct, dw = self.list_children[c]
        phys = ch.phys_of_type(ct, dw)
        out = []
        for k, cnt in enumerate(self.counts):
            ent = np.frombuffer(self.data[c][k], dtype=np.uint64).reshape(-1, 2)
            valid = np.unpackbits(self.validity[c][k].view(np.uint8), bitorder="little")[:cnt].astype(bool)
            raw = self.child_data[c][k]
            size = len(raw) // _out_width(ct, dw)
            cvalid = np.unpackbits(self.child_validity[c][k].view(np.uint8), bitorder="little")[:size].astype(bool)
            if phys == ch.P_STRING:
                e = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 16)
                vals = []
                for i in range(size):
                    ln = int(e[i, 0:4].view(np.uint32)[0])
                    b = bytes(e[i, 4:4 + ln]) if ln <= 12 else C.string_at(int(e[i, 8:16].view(np.uint64)[0]), ln)
                    vals.append(b.decode() if ct == ch.T_VARCHAR else b)
            elif phys in (ch.P_I128, ch.P_U128):
                vals = [int.from_bytes(raw[16 * i: 16 * i + 16], "little", signed=phys == ch.P_I128) for i in range(size)]
            else:
                vals = np.frombuffer(raw, dtype=_CHILD_DTYPE[phys]).tolist()
                if phys == ch.P_BOOL:
                    vals = [bool(v) for v in vals]
            for i in range(cnt):
                if not valid[i]:
                    out.append(None)
                    continue
                o, ln = int(ent[i, 0]), int(ent[i, 1])
                out.append([vals[j] if cvalid[j] else None for j in range(o, o + ln)])
        return out

    @property
    def nrows(self) -> int:
        return int(sum(self.counts))

    def column_bytes(self, c: int) -> bytes:
        return b"".join(self.data[c])

    def valid_bits(self, c: int) -> np.ndarray:
        """bool per row"""
        out = []
        for k, cnt in enumerate(self.counts):
            bits = np.unpackbits(self.validity[c][k].view(np.uint8), bitorder="little")[:cnt]
            out.append(bits.astype(bool))
        return np.concatenate(out) if out else np.zeros(0, dtype=bool)


class Appender:
    def __init__(self, ctx: GpuContext, type_ids: Sequence[int], sink: Optional[Callable] = None,
                 discard: bool = False):
        """`Connection::create_appender` (:955-971).  `discard=True`: no sink at all (conversion only,
        what bench.py's C5 measures: ingestion into one DuckDB appender is serial by libduckdb's design)."""
        self.lib = ctx.lib
        self.ctx = ctx
        self.type_ids = list(type_ids)
        self._sink_py = sink
        n = len(self.type_ids)

        def _trampoline(user, ncols, count, vec_data, vec_validity):
            try:
                return 1 if self._sink_py(int(count), [vec_data[i] for i in range(ncols)],
                                          [vec_validity[i] for i in range(ncols)]) else 0
            except Exception:  # noqa: BLE001 - a raising sink aborts the append
                return 0

        if isinstance(sink, CollectedChunks):
            sink.appender = self
        self._cb = nat.CHUNK_SINK(_trampoline) if (sink is not None and not discard) else nat.CHUNK_SINK()
        ids = (C.c_int32 * n)(*self.type_ids)
        self.handle = self.lib.duckdb_mb_gpu_appender_create(ctx.handle, n, ids, self._cb, None)
        if not self.handle:
            raise DuckDBError("create_appender failed: " + nat.last_error())

    # ---- protocol
    @property
    def state(self) -> int:
        return self.lib.duckdb_mb_gpu_appender_state(self.handle) if self.handle else CLOSED

    @property
    def row_count(self) -> int:
        return int(self.lib.duckdb_mb_gpu_appender_row_count(self.handle))

    @property
    def flushed_row_count(self) -> int:
        return int(self.lib.duckdb_mb_gpu_appender_flushed_row_count(self.handle))

    def error(self) -> str:  # appender_error, src/duckdb_native.c:1093-1098
        return nat.moonbit_bytes(self.lib.duckdb_mb_gpu_appender_error(self.handle)).decode(errors="replace")

    def _check(self, ok: int, what: str) -> None:
        if not ok:
            raise DuckDBError(self.error() or f"{what} failed")

    def begin_row(self):  # :974
        self._check(self.lib.duckdb_mb_gpu_begin_row(self.handle), "begin_row")

    def append_int(self, value: int):  # :983
        self._check(self.lib.duckdb_mb_gpu_append_int(self.handle, int(np.int32(value))), "append_int")

    def append_bigint(self, value: int):  # :995
        self._check(self.lib.duckdb_mb_gpu_append_bigint(self.handle, int(value)), "append_bigint")

    def append_double(self, value: float):  # :1007
        self._check(self.lib.duckdb_mb_gpu_append_double(self.handle, float(value)), "append_double")

    def append_varchar(self, value: str):  # :1019
        b = value.encode("utf-8") if isinstance(value, str) else bytes(value)
        self._check(self.lib.duckdb_mb_gpu_append_varchar(self.handle, b, len(b)), "append_varchar")

    def append_bool(self, value: bool):  # :1031
        self._check(self.lib.duckdb_mb_gpu_append_bool(self.handle, 1 if value else 0), "append_bool")

    def append_null(self):  # :1043
        self._check(self.lib.duckdb_mb_gpu_append_null(self.handle), "append_null")

    def append_date(self, days: int):
        self._check(self.lib.duckdb_mb_gpu_append_date(self.handle, int(days)), "append_date")

    def append_timestamp(self, micros: int):
        self._check(self.lib.duckdb_mb_gpu_append_timestamp(self.handle, int(micros)), "append_timestamp")

    def append_blob(self, data: bytes):  # src/duckdb_native.mbt:165-177 / src/duckdb_native.c:1397
        self._check(self.lib.duckdb_mb_gpu_append_blob(self.handle, data, len(data)), "append_blob")

    def set_decimal(self, col: int, width: int, scale: int):
        """The table column's DECIMAL(width, scale) (what duckdb_appender_column_type reports).  Arrow batches are
        converted to this width and must carry decimal128 at this scale with a precision <= width; without a declaration
        the first Arrow batch (or row-API value) declares it."""
        self._check(self.lib.duckdb_mb_gpu_appender_set_decimal(self.handle, int(col), int(width), int(scale)), "set_decimal")

    def set_list(self, col: int, child_type: int, dec_width: int = 0, dec_scale: int = 0):
        """The LIST column's child type (what duckdb_list_type_child_type of duckdb_appender_column_type reports);
        needed before an Arrow list reaches that column."""
        self._check(self.lib.duckdb_mb_gpu_appender_set_list(self.handle, int(col), int(child_type), int(dec_width), int(dec_scale)),
                    "set_list")

    def list_child(self, col: int):
        """Inside a sink call: (child values pointer, child mask pointer, child size) of LIST column `col`."""
        data, words, size = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self._check(self.lib.duckdb_mb_gpu_appender_list_child(self.handle, int(col), C.byref(data), C.byref(words), C.byref(size)),
                    "list_child")
        return data.value, words.value, int(size.value)

    def append_decimal(self, width: int, scale: int, unscaled: int):  # src/duckdb_native.c:1447-1481 (hugeint parts)
        lo = unscaled & 0xFFFFFFFFFFFFFFFF
        hi = (unscaled >> 64) & 0xFFFFFFFFFFFFFFFF
        as_i64 = lambda x: x - (1 << 64) if x >= (1 << 63) else x  # noqa: E731
        self._check(self.lib.duckdb_mb_gpu_append_decimal(self.handle, int(width), int(scale), as_i64(lo), as_i64(hi)), "append_decimal")

    def append_interval(self, months: int, days: int, micros: int):  # src/duckdb_native.c:1511-1533
        self._check(self.lib.duckdb_mb_gpu_append_interval(self.handle, int(months), int(days), int(micros)), "append_interval")

    @staticmethod
    def _bytes_array(items):
        """Array[Bytes] of the reference (moonbit_bytes_t* + lengths) as (pointer array, int32 lengths, keep-alive)"""
        enc = [x.encode("utf-8") if isinstance(x, str) else bytes(x) for x in items]
        bufs = [C.create_string_buffer(b, len(b) + 1) for b in enc]
        ptrs = (C.c_void_p * max(len(enc), 1))(*[C.addressof(b) for b in bufs])
        lens = (C.c_int32 * max(len(enc), 1))(*[len(b) for b in enc])
        return ptrs, lens, bufs

    def append_list_varchar(self, values):  # src/duckdb_native.mbt:1703-1715 / src/duckdb_native.c:1735-1790
        p, l, keep = self._bytes_array(values)
        self._check(self.lib.duckdb_mb_gpu_append_list_varchar(self.handle, p, l, len(values)), "append_list_varchar")

    def append_struct(self, fields, values):  # src/duckdb_native.mbt:1719-1735 / src/duckdb_native.c:1792-1858
        if len(fields) != len(values):
            raise ValueError("append_struct: fields and values differ in length")
        pn, ln, k1 = self._bytes_array(fields)
        pv, lv, k2 = self._bytes_array(values)
        self._check(self.lib.duckdb_mb_gpu_append_struct_varchar(self.handle, pn, ln, pv, lv, len(fields)), "append_struct")

    def append_map(self, keys, values):  # src/duckdb_native.mbt:1739-1755 / src/duckdb_native.c:1860-1926
        if len(keys) != len(values):
            raise ValueError("append_map: keys and values differ in length")
        pk, lk, k1 = self._bytes_array(keys)
        pv, lv, k2 = self._bytes_array(values)
        self._check(self.lib.duckdb_mb_gpu_append_map_varchar_varchar(self.handle, pk, lk, pv, lv, len(keys)), "append_map")

    def append_list_varchar_value(self, values):  # src/duckdb_native.mbt:1764-1795: a list literal, quotes doubled
        self.append_varchar("[" + ", ".join("'" + v.replace("'", "''") + "'" for v in values) + "]")

    def end_row(self):  # :1052
        self._check(self.lib.duckdb_mb_gpu_end_row(self.handle), "end_row")

    def flush(self):  # :1061
        self._check(self.lib.duckdb_mb_gpu_appender_flush(self.handle), "flush")

    def close(self):  # :1070-1076
        if self.handle:
            ok = self.lib.duckdb_mb_gpu_appender_close(self.handle)
            err = self.error() if not ok else ""
            self.lib.duckdb_mb_gpu_appender_destroy(self.handle)
            self.handle = None
            if not ok:
                raise DuckDBError(err or "close failed")

    # ---- additive bulk door
    def append_arrow(self, batch) -> None:
        """One pyarrow RecordBatch (or StructArray) -> DataChunks; legal where begin_row is."""
        import pyarrow as pa

        if isinstance(batch, pa.RecordBatch):
            batch = batch.to_struct_array()
        arr, sch = nat.ArrowArray(), nat.ArrowSchema()
        batch._export_to_c(C.addressof(arr), C.addressof(sch))
        try:
            ok = self.lib.duckdb_mb_gpu_append_arrow_batch(self.handle, C.addressof(arr), C.addressof(sch))
        finally:
            _release(arr)
            _release(sch)
        self._check(ok, "append_arrow_batch")

    def append_arrow_c(self, array_ptr: int, schema_ptr: int) -> None:
        self._check(self.lib.duckdb_mb_gpu_append_arrow_batch(self.handle, array_ptr, schema_ptr), "append_arrow_batch")

    def timings(self) -> dict:
        t = (C.c_double * 4)()
        b = (C.c_uint64 * 2)()
        self.lib.duckdb_mb_gpu_appender_timings(self.handle, t)
        self.lib.duckdb_mb_gpu_appender_link_bytes(self.handle, b)
        return {"h2d_ms": t[0], "kernels_ms": t[1], "d2h_ms": t[2], "total_ms": t[3], "h2d_bytes": b[0], "d2h_bytes": b[1]}


_RELEASE = C.CFUNCTYPE(None, C.c_void_p)


def _release(obj) -> None:
    """Call the release callback of an exported ArrowArray / ArrowSchema (consumer's duty)."""
    if obj.release:
        _RELEASE(obj.release)(C.addressof(obj))


# ---- the pure model (src/duckdb_appender_state_machine.mbt:7-239), used to cross-check the C side
class AppenderModel:
    def __init__(self, expected_columns: int):
        self.state = NOT_CREATED
        self.column_count = 0
        self.expected_columns = expected_columns
        self.row_count = 0
        self.flushed_row_count = 0

    def execute(self, cmd: str) -> "AppenderModel":
        s = self.state
        if s == CLOSED:
            return self
        if s == ERROR:
            if cmd == "close":
                self.state = CLOSED
            return self
        if s == NOT_CREATED and cmd == "create":
            self.state, self.column_count, self.row_count, self.flushed_row_count = READY, 0, 0, 0
        elif s in (READY, FLUSHED) and cmd == "begin_row":
            self.state, self.column_count = ROW_IN_PROGRESS, 0
        elif s in (READY, FLUSHED) and cmd == "flush":
            self.state, self.column_count, self.flushed_row_count = FLUSHED, 0, self.row_count
        elif s in (READY, FLUSHED, ROW_IN_PROGRESS) and cmd == "close":
            self.state = CLOSED
        elif s == ROW_IN_PROGRESS and cmd.startswith("append"):
            if self.column_count < self.expected_columns:
                self.column_count += 1
            else:
                self.state = ERROR
        elif s == ROW_IN_PROGRESS and cmd == "end_row":
            if self.column_count == self.expected_columns:
                self.state, self.column_count, self.row_count = READY, 0, self.row_count + 1
            else:
                self.state = ERROR
        else:
            self.state = ERROR
        return self
