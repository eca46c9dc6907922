"""Plain-Python statement of what a DuckDB table column holds after an Arrow array is appended to it, and a plain
decoder of the DataChunk vectors the appender hands to its sink.  Independent of oracle/oracle.c and of the kernels.

Expected cells read the Arrow values through pyarrow's own decoding (`to_pylist`, `datetime`, `decimal.Decimal`).  The
raw Arrow buffer is read only where Python would lose information: FLOAT / DOUBLE bit patterns (`to_pylist` widens a
float32 and quiets a signalling NaN) and temporal values outside `datetime`'s range or below its microsecond unit.
The decoder reads the vectors with `struct` / `int.from_bytes` only and asserts the vector-level invariants the
project promises.  The only thing taken from the code under test is the set of type ids in `chunks.py`.

Cell values, one form per column type:
  integers, DATE (days), TIME / TIME_NS / TIMESTAMP* (ticks of the column's unit), DECIMAL (the unscaled integer at the
  table's scale), HUGEINT: int;  FLOAT / DOUBLE: the IEEE bit pattern as an unsigned int;  BOOLEAN: the byte, 0 or 1;
  VARCHAR / BLOB: bytes;  UHUGEINT / UUID: the 16 stored bytes;  TIME_TZ: the stored uint64.

Deviation from DuckDB semantics, kept on purpose: UHUGEINT and UUID columns take an Arrow `fixed_size_binary(16)`
('w:16') and TIME_TZ takes a uint64 ('L'), all as DuckDB's stored bytes, unchanged.  That is this project's contract
in both directions (the forward path exports those columns the same way).  In particular a UUID here is DuckDB's
hugeint with the top bit flipped, not the RFC 4122 bytes of Arrow's `arrow.uuid` extension type.
"""
from __future__ import annotations

import ctypes
import datetime
import struct
from decimal import Decimal
from typing import Callable, List, Optional

from duckdb_mbt_b200 import chunks as ch

VECTOR_SIZE = 2048
I32_MAX = 2**31 - 1

UNSIGNED = {ch.T_UTINYINT: 8, ch.T_USMALLINT: 16, ch.T_UINTEGER: 32, ch.T_UBIGINT: 64}
SIGNED = {ch.T_TINYINT: 8, ch.T_SMALLINT: 16, ch.T_INTEGER: 32, ch.T_BIGINT: 64}
TIMESTAMPS = {ch.T_TIMESTAMP: 10**6, ch.T_TIMESTAMP_TZ: 10**6, ch.T_TIMESTAMP_S: 1, ch.T_TIMESTAMP_MS: 10**3, ch.T_TIMESTAMP_NS: 10**9}
STRINGS = (ch.T_VARCHAR, ch.T_BLOB)
RAW16 = (ch.T_UHUGEINT, ch.T_UUID)  # the deviation above


def decimal_width_bytes(width: int) -> int:
    """DuckDB's physical storage of DECIMAL(width, s): int16 / int32 / int64 / int128"""
    return 2 if width <= 4 else 4 if width <= 9 else 8 if width <= 18 else 16


def vector_width(type_id: int, dec_width: int = 0) -> int:
    """bytes per row of a DuckDB vector of this type"""
    if type_id in SIGNED:
        return SIGNED[type_id] // 8
    if type_id in UNSIGNED:
        return UNSIGNED[type_id] // 8
    if type_id == ch.T_DECIMAL:
        return decimal_width_bytes(dec_width)
    if type_id == ch.T_BOOLEAN:
        return 1
    if type_id in (ch.T_FLOAT, ch.T_DATE):
        return 4
    if type_id in (ch.T_DOUBLE, ch.T_TIME, ch.T_TIME_NS, ch.T_TIME_TZ) or type_id in TIMESTAMPS:
        return 8
    if type_id in (ch.T_HUGEINT, ch.T_LIST) or type_id in STRINGS or type_id in RAW16:
        return 16
    raise KeyError(type_id)


# ---------------------------------------------------------------- what DuckDB stores
def unscaled(d: Decimal, scale: int) -> int:
    """the integer d * 10^scale, exactly (no context rounding); raises if d has more fractional digits than scale"""
    sign, digits, exp = d.as_tuple()
    n = int("".join(map(str, digits)) or "0")
    e = exp + scale
    if e < 0:
        q, r = divmod(n, 10 ** -e)
        if r:
            raise ValueError(f"{d} has more than {scale} fractional digits")
        n = q
    else:
        n *= 10 ** e
    return -n if sign else n


def decimal_refusal(precision: int, scale: int, bit_width: int, type_id: int, table: Optional[tuple]) -> Optional[str]:
    """Why an Arrow decimal<bit_width>(precision, scale) cannot go into the column (None: it can).  A DECIMAL column
    holds DECIMAL(w, s) = `table` (None: not declared, the Arrow type declares it); HUGEINT is DECIMAL(38, 0).  The
    project refuses rather than casts: the values keep their unscaled integers, so the scale must be the table's, and
    every value within the Arrow precision must fit the table's width."""
    if bit_width != 128:
        return f"{bit_width}-bit"
    w, s = (38, 0) if type_id == ch.T_HUGEINT else (table or (precision, scale))
    if scale != s:
        return "scale"
    if precision > w:
        return "precision"
    return None


def _raw_ints(arr, fmt: str) -> List[int]:
    """the raw values of a fixed-width Arrow array (ignoring validity)"""
    size = struct.calcsize(fmt)
    buf = arr.buffers()[1]
    return [v for (v,) in struct.iter_unpack("<" + fmt, bytes(buf)[arr.offset * size:(arr.offset + len(arr)) * size])]


def _ticks(v, per_sec: int) -> int:
    """a datetime / time as ticks of 1/per_sec second since the epoch / midnight, exact integer arithmetic"""
    if isinstance(v, datetime.time):
        us = ((v.hour * 60 + v.minute) * 60 + v.second) * 10**6 + v.microsecond
    else:
        epoch = datetime.datetime(1970, 1, 1, tzinfo=datetime.timezone.utc if v.tzinfo else None)
        us = (v - epoch) // datetime.timedelta(microseconds=1)
    assert (us * per_sec) % 10**6 == 0
    return us * per_sec // 10**6


# what datetime holds, in ticks of each unit: date, time of day (no 24:00:00), datetime from 0001-01-01 to 9999-12-31
DATE_RANGE = (-719162, 2932896)
TIME_RANGE_US = (0, 86_400 * 10**6 - 1)
DATETIME_RANGE_US = (-62135596800 * 10**6, 253402300799 * 10**6 + 999_999)


def _python_values(arr, raw: List[int], lo: int, hi: int) -> list:
    """`to_pylist` of the rows whose raw value lies in [lo, hi], the range Python's type holds; None elsewhere"""
    ok = [lo <= r <= hi for r in raw]
    vals = iter(arr.filter(ok).to_pylist())
    return [next(vals) if k else None for k in ok]


def expected_cells(arr, type_id: int, table_decimal: Optional[tuple] = None) -> list:
    """the value DuckDB holds in each row after `arr` (a pyarrow array) is appended to a column of `type_id`;
    None for NULL.  `table_decimal`: the DECIMAL column's (width, scale)."""
    valid = arr.is_valid().to_pylist() if arr.null_count else [True] * len(arr)

    def mask(vals):
        return [v if ok else None for v, ok in zip(vals, valid)]

    if type_id in (ch.T_FLOAT, ch.T_DOUBLE):
        return mask(_raw_ints(arr, "I" if type_id == ch.T_FLOAT else "Q"))
    if type_id == ch.T_TIME_TZ:
        return mask(_raw_ints(arr, "Q"))
    if type_id == ch.T_DATE:
        raw = _raw_ints(arr, "i")
        py = _python_values(arr, raw, *DATE_RANGE)
        # outside datetime.date (DuckDB's +-infinity among them): the day number itself
        return mask([(v - datetime.date(1970, 1, 1)).days if v is not None else r for v, r in zip(py, raw)])
    if type_id in TIMESTAMPS or type_id in (ch.T_TIME, ch.T_TIME_NS):
        per_sec = TIMESTAMPS.get(type_id) or (10**9 if type_id == ch.T_TIME_NS else 10**6)
        raw = _raw_ints(arr, "q")
        if per_sec > 10**6:  # below datetime's microsecond: the raw ticks
            return mask(raw)
        if getattr(arr.type, "tz", None):  # the same instants as naive UTC datetimes, which are much cheaper to build
            import pyarrow as pa
            arr = arr.cast(pa.timestamp(arr.type.unit))
        # datetime.time has no 24:00:00 (DuckDB's end of day): pyarrow would wrap it to 00:00
        lo, hi = TIME_RANGE_US if type_id == ch.T_TIME else DATETIME_RANGE_US
        py = _python_values(arr, raw, -(-lo * per_sec // 10**6), hi * per_sec // 10**6)
        return mask([_ticks(v, per_sec) if v is not None else r for v, r in zip(py, raw)])
    py = arr.to_pylist()
    if type_id == ch.T_BOOLEAN:
        return [None if v is None else int(v) for v in py]
    if type_id == ch.T_DECIMAL:
        scale = table_decimal[1] if table_decimal else arr.type.scale
        return [None if v is None else unscaled(v, scale) for v in py]
    if type_id == ch.T_HUGEINT:
        return [None if v is None else unscaled(v, 0) for v in py]
    if type_id in STRINGS:
        return [None if v is None else (v.encode() if isinstance(v, str) else bytes(v)) for v in py]
    if type_id in RAW16:
        return [None if v is None else bytes(v) for v in py]
    if type_id in SIGNED or type_id in UNSIGNED:
        return py
    raise KeyError(type_id)


def expected_lists(arr, child_type: int, table_decimal: Optional[tuple] = None) -> list:
    """a pyarrow list / large_list array -> per row None or the list of expected child cells"""
    values = expected_cells(arr.values, child_type, table_decimal)  # the whole child array, offsets index into it
    offs = arr.offsets.to_pylist()
    valid = arr.is_valid().to_pylist()
    return [[*values[offs[i]:offs[i + 1]]] if valid[i] else None for i in range(len(arr))]


# ---------------------------------------------------------------- decoding the vectors a sink received
def _bit(words: bytes, i: int) -> bool:
    return bool(words[i >> 3] >> (i & 7) & 1)


def decode_vector(data: bytes, validity: Optional[bytes], count: int, type_id: int, dec_width: int = 0,
                  deref: Callable[[int, int], bytes] = ctypes.string_at, strict: bool = True) -> list:
    """One vector of `count` rows -> per row a cell value (the forms of `expected_cells`) or None.  `validity`: the
    uint64 mask words as bytes, None for all-valid.  `strict`: also hold the sink-side promises (NULL payload bytes
    zero, validity bits past `count` zero); a table that copied the vector (DuckDB, the mock) keeps neither."""
    w = vector_width(type_id, dec_width)
    assert len(data) >= count * w
    if strict and validity is not None:
        assert not any(_bit(validity, i) for i in range(count, 8 * len(validity))), "validity bits past count"
    out = []
    for i in range(count):
        cell = data[i * w:(i + 1) * w]
        if validity is not None and not _bit(validity, i):
            if strict and type_id != ch.T_LIST:
                assert cell == bytes(w), f"row {i}: NULL payload {cell.hex()}"
            out.append(None)
            continue
        out.append(decode_cell(cell, type_id, deref))
    return out


def decode_cell(cell: bytes, type_id: int, deref: Callable[[int, int], bytes] = ctypes.string_at):
    if type_id in SIGNED or type_id in (ch.T_DATE, ch.T_TIME, ch.T_TIME_NS, ch.T_DECIMAL, ch.T_HUGEINT) or type_id in TIMESTAMPS:
        return int.from_bytes(cell, "little", signed=True)
    if type_id in UNSIGNED or type_id in (ch.T_FLOAT, ch.T_DOUBLE, ch.T_TIME_TZ):
        return int.from_bytes(cell, "little", signed=False)
    if type_id == ch.T_BOOLEAN:
        assert cell[0] in (0, 1), f"BOOLEAN byte {cell[0]}"
        return cell[0]
    if type_id in RAW16:
        return bytes(cell)
    if type_id in STRINGS:
        (length,) = struct.unpack_from("<I", cell, 0)
        if length <= 12:
            assert cell[4 + length:] == bytes(12 - length), f"inline string_t padding {cell.hex()}"
            return bytes(cell[4:4 + length])
        (ptr,) = struct.unpack_from("<Q", cell, 8)
        s = deref(ptr, length)
        assert cell[4:8] == s[:4], f"string_t prefix {cell[4:8].hex()} of {s[:8].hex()}"
        return s
    raise KeyError(type_id)


def decode_list_vector(entries: bytes, validity: Optional[bytes], count: int, child: bytes, child_validity: Optional[bytes],
                       child_size: int, child_type: int, dec_width: int = 0, deref=ctypes.string_at, strict: bool = True) -> list:
    """a LIST vector (duckdb_list_entry {offset, length} per row) and its child vector -> per row None or a list"""
    cells = decode_vector(child, child_validity, child_size, child_type, dec_width, deref, strict)
    out = []
    for i in range(count):
        off, ln = struct.unpack_from("<QQ", entries, 16 * i)
        if validity is not None and not _bit(validity, i):
            if strict:
                assert ln == 0, f"row {i}: NULL list with length {ln}"
            out.append(None)
            continue
        assert off + ln <= child_size, f"row {i}: entry ({off}, {ln}) leaves the child vector of {child_size}"
        out.append(cells[off:off + ln])
    return out


def decode_collected(sink, col: int, type_id: int, dec_width: int = 0, child: Optional[tuple] = None) -> list:
    """every row of column `col` of a CollectedChunks sink; `child`: a LIST column's (child type, child dec width)"""
    out = []
    for k, count in enumerate(sink.counts):
        validity = bytes(sink.validity[col][k].tobytes())
        if type_id == ch.T_LIST:
            ct, dw = child
            raw = sink.child_data[col][k]
            size = len(raw) // vector_width(ct, dw)
            out += decode_list_vector(sink.data[col][k], validity, count, raw, bytes(sink.child_validity[col][k].tobytes()),
                                      size, ct, dw)
        else:
            out += decode_vector(sink.data[col][k], validity, count, type_id, dec_width)
    return out
