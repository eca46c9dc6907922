"""ctypes loader for the CPU oracle (oracle/oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this package; the product path (duckdb.mbt_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _LIB_PATH


class OraColumn(C.Structure):
    _fields_ = [("type_id", C.c_int32), ("phys", C.c_int32), ("dec_width", C.c_int32), ("dec_scale", C.c_int32),
                ("data", C.c_void_p), ("data_off", C.c_void_p), ("validity", C.c_void_p), ("val_off", C.c_void_p),
                ("name", C.c_char_p), ("dict_offsets", C.c_void_p), ("dict_data", C.c_void_p), ("dict_size", C.c_uint32)]


class OraBatch(C.Structure):
    _fields_ = [("nchunks", C.c_int64), ("counts", C.c_void_p), ("ncols", C.c_int32), ("cols", C.POINTER(OraColumn))]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        L.ora_result_create.restype = C.c_void_p
        L.ora_result_create.argtypes = [C.POINTER(OraBatch)]
        L.ora_result_destroy.argtypes = [C.c_void_p]
        L.ora_result_rows.restype = C.c_int64
        L.ora_result_rows.argtypes = [C.c_void_p]
        for name in ("int32", "int64", "double", "string", "bool"):
            for suffix in ("", "_nullable"):
                f = getattr(L, f"ora_arrow_get_column_{name}{suffix}")
                f.restype = C.c_void_p
                f.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int64)]
        L.ora_arrow_schema.restype = C.c_void_p
        L.ora_arrow_schema.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.ora_free.argtypes = [C.c_void_p]
        L.ora_value_is_null.restype = C.c_int
        L.ora_value_is_null.argtypes = [C.c_void_p, C.c_int32, C.c_int64]
        L.ora_value_varchar.restype = C.c_void_p
        L.ora_value_varchar.argtypes = [C.c_void_p, C.c_int32, C.c_int64]
        L.ora_arrow_fixed.restype = C.c_int
        L.ora_arrow_fixed.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
        L.ora_arrow_string.restype = C.c_int
        L.ora_arrow_string.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
        L.ora_typed_fixed_column.restype = C.c_int
        L.ora_typed_fixed_column.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ora_typed_from_text.restype = C.c_int
        L.ora_typed_from_text.argtypes = [C.c_int32, C.c_char_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
        L.ora_parse_int.restype = C.c_int32
        L.ora_parse_int.argtypes = [C.c_char_p, C.c_int64]
        L.ora_parse_double.restype = C.c_double
        L.ora_parse_double.argtypes = [C.c_char_p, C.c_int64]
        L.ora_parse_date.restype = C.c_int32
        L.ora_parse_date.argtypes = [C.c_char_p, C.c_int64, C.POINTER(C.c_int)]
        L.ora_parse_timestamp.restype = C.c_int64
        L.ora_parse_timestamp.argtypes = [C.c_char_p, C.c_int64, C.POINTER(C.c_int)]
        L.ora_date_to_days.restype = C.c_int32
        L.ora_date_to_days.argtypes = [C.c_int32, C.c_int32, C.c_int32]
        L.ora_render_date.restype = C.c_int
        L.ora_render_date.argtypes = [C.c_int32, C.c_char_p]
        L.ora_render_timestamp.restype = C.c_int
        L.ora_render_timestamp.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_char_p]
        L.ora_render_decimal64.restype = C.c_int
        L.ora_render_decimal64.argtypes = [C.c_int64, C.c_int, C.c_char_p]
        L.ora_render_double.restype = C.c_int
        L.ora_render_double.argtypes = [C.c_double, C.c_char_p]
        L.ora_render_float.restype = C.c_int
        L.ora_render_float.argtypes = [C.c_float, C.c_char_p]
        for name, vt in (("int32", None), ("int64_as_int", None), ("double", None), ("bool", None)):
            f = getattr(L, f"ora_decode_{name}")
            f.restype = C.c_int64
            f.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
        L.ora_decode_string.restype = C.c_int64
        L.ora_decode_string.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ora_rev_fixed.restype = C.c_int
        L.ora_rev_fixed.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
        L.ora_rev_string.restype = C.c_int
        L.ora_rev_string.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int64, C.c_int64,
                                     C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
        _lib = L
    return _lib


def _ptr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


class OracleResult:
    """The reference's `duckdb_mb_arrow_result` over a host ChunkBatch (anything with .counts and
    .columns carrying numpy slabs: see duckdb.mbt_b200/chunks.py)."""

    def __init__(self, batch):
        self._batch = batch  # keeps the numpy buffers alive
        L = lib()
        self._counts = np.ascontiguousarray(batch.counts, dtype=np.uint32)
        n = len(batch.columns)
        self._cols = (OraColumn * max(n, 1))()
        self._names = []
        for i, c in enumerate(batch.columns):
            nm = c.name.encode()
            self._names.append(nm)
            d_offs = d_data = None
            labels = getattr(c, "dictionary", None)
            if labels is not None:  # ENUM
                d_offs = np.zeros(len(labels) + 1, dtype=np.uint32)
                np.cumsum([len(x) for x in labels], out=d_offs[1:])
                d_data = np.frombuffer(b"".join(labels) + b"\0", dtype=np.uint8).copy()
                self._names.append((d_offs, d_data))
            self._cols[i] = OraColumn(c.type_id, c.phys, c.dec_width, c.dec_scale, _ptr(c.data), _ptr(c.data_off),
                                      _ptr(c.validity), _ptr(c.val_off), nm, _ptr(d_offs), _ptr(d_data),
                                      0 if labels is None else len(labels))
        self._b = OraBatch(self._counts.shape[0], _ptr(self._counts), n, self._cols)
        self.handle = L.ora_result_create(C.byref(self._b))
        self.nrows = int(L.ora_result_rows(self.handle))

    def close(self):
        if self.handle:
            lib().ora_result_destroy(self.handle)
            self.handle = None

    def __del__(self):
        self.close()

    # ---- reference packed getters (src/duckdb_native.c:2357-2797) -> bytes
    def _getter(self, name: str, col: int) -> bytes:
        L = lib()
        n = C.c_int64(0)
        p = getattr(L, name)(self.handle, col, C.byref(n))
        try:
            return C.string_at(p, n.value) if n.value > 0 else b""
        finally:
            L.ora_free(p)

    def get_column(self, kind: str, col: int, nullable: bool = False) -> bytes:
        return self._getter(f"ora_arrow_get_column_{kind}{'_nullable' if nullable else ''}", col)

    def cell_is_null(self, col: int, row: int) -> bool:
        """duckdb_mb_result_is_null (src/duckdb_native.c:215-222)"""
        return bool(lib().ora_value_is_null(self.handle, col, row))

    def cell_value(self, col: int, row: int) -> bytes:
        """duckdb_mb_result_value (src/duckdb_native.c:224-238): duckdb_value_varchar, empty Bytes for NULL"""
        p = lib().ora_value_varchar(self.handle, col, row)
        if not p:
            return b""
        out = C.string_at(p)
        lib().ora_free(p)
        return out

    def schema(self) -> bytes:
        L = lib()
        n = C.c_int64(0)
        p = L.ora_arrow_schema(self.handle, C.byref(n))
        try:
            return C.string_at(p, n.value)
        finally:
            L.ora_free(p)

    # ---- Arrow-layout oracle
    def arrow_fixed(self, col: int, dst: int, out_width: int, want_values: bool = True):
        """-> (values uint8[n*out_width] | bit-packed, bitmap uint8, valid_bytes uint8[n], null_count)"""
        n = self.nrows
        if dst == 5:  # BOOL_BITS
            values = np.zeros((n + 7) // 8, dtype=np.uint8)
        else:
            values = np.zeros(n * out_width, dtype=np.uint8)
        bitmap = np.zeros((n + 63) // 64 * 8, dtype=np.uint8)
        vbytes = np.zeros(n, dtype=np.uint8)
        nc = C.c_int64(0)
        rc = lib().ora_arrow_fixed(self.handle, col, dst, _ptr(values) if want_values else None, _ptr(bitmap),
                                   _ptr(vbytes), C.byref(nc))
        if rc != 0:
            raise ValueError("oracle: unsupported conversion")
        return values, bitmap, vbytes, nc.value

    def arrow_string(self, col: int, mode: int = 0):
        """-> (offsets int32|int64 [n+1], data uint8[total])"""
        n = self.nrows
        total = C.c_int64(0)
        lib().ora_arrow_string(self.handle, col, mode, None, None, C.byref(total))
        offsets = np.zeros(n + 1, dtype=np.int64 if mode == 1 else np.int32)
        data = np.zeros(total.value, dtype=np.uint8)
        rc = lib().ora_arrow_string(self.handle, col, mode, _ptr(offsets), _ptr(data) if total.value else None, C.byref(total))
        if rc != 0:
            raise ValueError("oracle: not a string column")
        return offsets, data

    def typed_fixed(self, col: int):
        """text round trip of the reference: -> (tags uint8[n], ivals int64[n], dvals float64[n])"""
        n = self.nrows
        tags = np.zeros(n, dtype=np.uint8)
        iv = np.zeros(n, dtype=np.int64)
        dv = np.zeros(n, dtype=np.float64)
        rc = lib().ora_typed_fixed_column(self.handle, col, _ptr(tags), _ptr(iv), _ptr(dv))
        if rc != 0:
            raise ValueError("oracle: no text renderer for this column type")
        return tags, iv, dv


# ---- MoonBit decoders (src/duckdb_arrow_native.mbt:430-822)
def decode_int32(blob: bytes, nullable: bool = False):
    n = max(len(blob), 1)
    buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    values = np.zeros(n, dtype=np.int32)
    valid = np.zeros(n, dtype=np.uint8)
    c = lib().ora_decode_int32(_ptr(buf), len(blob), int(nullable), _ptr(values), _ptr(valid))
    return values[:c].copy(), valid[:c].astype(bool)


def decode_int64_as_int(blob: bytes, nullable: bool = False):
    n = max(len(blob), 1)
    buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    values = np.zeros(n, dtype=np.int32)
    valid = np.zeros(n, dtype=np.uint8)
    c = lib().ora_decode_int64_as_int(_ptr(buf), len(blob), int(nullable), _ptr(values), _ptr(valid))
    return values[:c].copy(), valid[:c].astype(bool)


def decode_double(blob: bytes, nullable: bool = False):
    n = max(len(blob), 1)
    buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    values = np.zeros(n, dtype=np.float64)
    valid = np.zeros(n, dtype=np.uint8)
    c = lib().ora_decode_double(_ptr(buf), len(blob), int(nullable), _ptr(values), _ptr(valid))
    return values[:c].copy(), valid[:c].astype(bool)


def decode_bool(blob: bytes, nullable: bool = False):
    n = max(len(blob), 1)
    buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    values = np.zeros(n, dtype=np.uint8)
    valid = np.zeros(n, dtype=np.uint8)
    c = lib().ora_decode_bool(_ptr(buf), len(blob), int(nullable), _ptr(values), _ptr(valid))
    return values[:c].astype(bool), valid[:c].astype(bool)


def decode_string(blob: bytes, nullable: bool = False) -> Tuple[List[bytes], np.ndarray]:
    n = max(len(blob), 1)
    buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    starts = np.zeros(n, dtype=np.int64)
    ends = np.zeros(n, dtype=np.int64)
    valid = np.zeros(n, dtype=np.uint8)
    c = lib().ora_decode_string(_ptr(buf), len(blob), int(nullable), _ptr(starts), _ptr(ends), _ptr(valid))
    return [blob[starts[i]:ends[i]] for i in range(c)], valid[:c].astype(bool)


def parse_int(s: str) -> int:
    b = s.encode()
    return int(lib().ora_parse_int(b, len(b)))


def parse_double(s: str) -> float:
    b = s.encode()
    return float(lib().ora_parse_double(b, len(b)))


def parse_date(s: str) -> Optional[int]:
    b = s.encode()
    ok = C.c_int(0)
    v = lib().ora_parse_date(b, len(b), C.byref(ok))
    return int(v) if ok.value else None


def parse_timestamp(s: str) -> Optional[int]:
    b = s.encode()
    ok = C.c_int(0)
    v = lib().ora_parse_timestamp(b, len(b), C.byref(ok))
    return int(v) if ok.value else None


def typed_from_text(type_id: int, s: str):
    """parse_value_with_type (src/duckdb_parsing.mbt:82-144) -> (tag, value)"""
    b = s.encode()
    iv, dv = C.c_int64(0), C.c_double(0.0)
    tag = lib().ora_typed_from_text(type_id, b, len(b), C.byref(iv), C.byref(dv))
    if tag == 1:
        return tag, dv.value
    if tag == 3:
        return tag, s
    return tag, iv.value


def _render(fn, *args) -> str:
    buf = C.create_string_buffer(128)
    n = fn(*args, buf)
    return buf.raw[:n].decode()


def render_date(days: int) -> str:
    return _render(lib().ora_render_date, days)


def render_timestamp(v: int, unit_per_sec: int = 1_000_000, tz: bool = False) -> str:
    return _render(lib().ora_render_timestamp, v, unit_per_sec, int(tz))


def render_decimal64(v: int, scale: int) -> str:
    return _render(lib().ora_render_decimal64, v, scale)


def render_double(v: float) -> str:
    return _render(lib().ora_render_double, v)


def render_float(v: float) -> str:
    return _render(lib().ora_render_float, v)


def rev_fixed(values: np.ndarray, bitmap: Optional[np.ndarray], bit_offset: int, nrows: int, rev_op: int, w_out: int):
    nchunks = (nrows + 2047) // 2048
    out = np.zeros(max(nchunks, 1) * 2048 * w_out, dtype=np.uint8)
    val = np.zeros(max(nchunks, 1) * 32, dtype=np.uint64)
    nc = C.c_int64(0)
    lib().ora_rev_fixed(_ptr(values), _ptr(bitmap), bit_offset, nrows, rev_op, _ptr(out), _ptr(val), C.byref(nc))
    return out, val, nc.value


def rev_string(offsets: np.ndarray, data: np.ndarray, data_host_base: int, bitmap: Optional[np.ndarray],
               bit_offset: int, nrows: int):
    nchunks = (nrows + 2047) // 2048
    out = np.zeros(max(nchunks, 1) * 2048 * 16, dtype=np.uint8)
    val = np.zeros(max(nchunks, 1) * 32, dtype=np.uint64)
    nc = C.c_int64(0)
    large = 1 if offsets.dtype == np.int64 else 0
    lib().ora_rev_string(_ptr(offsets), large, _ptr(data), data_host_base, _ptr(bitmap), bit_offset, nrows,
                         _ptr(out), _ptr(val), C.byref(nc))
    return out, val, nc.value


def _bytes_array(items):
    enc = [x.encode("utf-8") if isinstance(x, str) else bytes(x) for x in items]
    bufs = [C.create_string_buffer(b, len(b) + 1) for b in enc]
    ptrs = (C.c_void_p * max(len(enc), 1))(*[C.addressof(b) for b in bufs])
    lens = (C.c_int32 * max(len(enc), 1))(*[len(b) for b in enc])
    return ptrs, lens, bufs, sum(len(b) for b in enc)


def list_varchar_text(values) -> bytes:
    """the VARCHAR cell duckdb_mb_append_list_varchar appends (src/duckdb_native.c:1735-1790)"""
    p, l, keep, total = _bytes_array(values)
    out = C.create_string_buffer(total + 4 * len(values) + 8)
    f = lib().ora_list_varchar_text
    f.restype = C.c_int64
    n = f(p, l, C.c_int32(len(values)), out)
    return out.raw[:n]


def pairs_varchar_text(keys, values) -> bytes:
    """the VARCHAR cell duckdb_mb_append_struct_varchar / _map_varchar_varchar append (:1792-1926)"""
    pk, lk, k1, t1 = _bytes_array(keys)
    pv, lv, k2, t2 = _bytes_array(values)
    out = C.create_string_buffer(t1 + t2 + 8 * len(keys) + 8)
    f = lib().ora_pairs_varchar_text
    f.restype = C.c_int64
    n = f(pk, lk, pv, lv, C.c_int32(len(keys)), out)
    return out.raw[:n]


def list_arrow(entries: np.ndarray, data_off: np.ndarray, validity: Optional[np.ndarray], val_off: np.ndarray,
               counts: np.ndarray, child_base: np.ndarray, child_data: np.ndarray, child_validity: Optional[np.ndarray],
               child_val_off: Optional[np.ndarray], child_width: int, large: bool, capacity: int):
    """LIST vectors -> Arrow list<child>: (offsets, child bytes, child bitmap bytes, total, child null count)"""
    nrows = int(np.asarray(counts, dtype=np.int64).sum())
    offsets = np.zeros(nrows + 1, dtype=np.int64 if large else np.int32)
    child = np.zeros(max(capacity, 1) * child_width, dtype=np.uint8)
    bitmap = np.zeros((max(capacity, 1) + 63) // 64 * 8 + 8, dtype=np.uint8)
    total, nulls = C.c_int64(0), C.c_int64(0)
    f = lib().ora_list_arrow
    f.restype = C.c_int
    f.argtypes = [C.c_void_p] * 5 + [C.c_int64] + [C.c_void_p] * 4 + [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.POINTER(C.c_int64)] * 2
    f(_ptr(entries), _ptr(data_off), _ptr(validity), _ptr(val_off), _ptr(np.ascontiguousarray(counts, dtype=np.uint32)),
      int(len(counts)), _ptr(child_base), _ptr(child_data), _ptr(child_validity), _ptr(child_val_off), child_width,
      1 if large else 0, _ptr(offsets), _ptr(child), _ptr(bitmap), C.byref(total), C.byref(nulls))
    return offsets, child[: total.value * child_width], bitmap, total.value, nulls.value
