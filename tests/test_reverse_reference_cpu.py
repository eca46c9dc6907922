"""CPU: tests/reverse_semantics.py against hand-written known answers; the CPU oracle's reverse conversions
(ora_rev_fixed / ora_rev_string) against it for the op the *table* type implies; and the placement the GPU tests use
(tests/test_gpu_append_reference.py), pinned so that every edge value reaches every position that matters to the
reverse kernels.

The edge sets, the (Arrow type, column type) pairs the appender accepts and the placement live here so that the GPU
file imports them."""
import ctypes
import math
import struct
from decimal import Decimal

import numpy as np
import pytest

pa = pytest.importorskip("pyarrow")

import reverse_semantics as rs  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402

I64_MIN, I64_MAX = -2**63, 2**63 - 1

# ---------------------------------------------------------------------------------------------- edge sets
def _int_edges(bits: int, signed: bool) -> list:
    lo, hi = (-2**(bits - 1), 2**(bits - 1) - 1) if signed else (0, 2**bits - 1)
    return sorted({lo, lo + 1, -1 if signed else 2, 0, 1, hi - 1, hi})


F32_BITS = [0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0x7FA00005, 0xFFA0BEEF, 0x00000001, 0x80000001,
            0x7F7FFFFF, 0xFF7FFFFF, 0x3F800000]
F64_BITS = [0x0, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000, 0x7FF8000000000000, 0x7FF4000000000005,
            0xFFF00000DEADBEEF, 0x1, 0x8000000000000001, 0x7FEFFFFFFFFFFFFF, 0xFFEFFFFFFFFFFFFF, 0x3FF0000000000000]
DATE_EDGES = [rs.I32_MAX, -rs.I32_MAX, -719162, 2932896, 0, -1, 1]  # datetime.date's limits: 0001-01-01, 9999-12-31
TIME_EDGES = {"us": [0, 1, 86_399_999_999, 86_400_000_000], "ns": [0, 1, 86_399_999_999_999, 86_400_000_000_000]}
_DT_MIN_US, _DT_MAX_US = -62135596800 * 10**6, 253402300799 * 10**6 + 999999  # datetime's range in microseconds


def _ts_edges(unit: str) -> list:
    per_us = {"s": None, "ms": None, "us": 1, "ns": 1000}[unit]
    extra = []
    if unit == "s":
        extra = [_DT_MIN_US // 10**6, _DT_MAX_US // 10**6]
    elif unit == "ms":
        extra = [_DT_MIN_US // 1000, _DT_MAX_US // 1000]
    elif per_us == 1:
        extra = [_DT_MIN_US, _DT_MAX_US]
    return [I64_MAX, -I64_MAX, I64_MIN + 1, 0, -1, 1, 1_700_000_000_123_456] + extra


def decimal_values(p: int, s: int) -> list:
    """+-(10^p - 1), +-10^(p-1), +-1, 0 as unscaled integers of DECIMAL(p, s)"""
    return [Decimal(v).scaleb(-s) for v in (10**p - 1, -(10**p - 1), 10**(p - 1), -10**(p - 1), 1, -1, 0)]


BIG = 70 * 1024


def string_edges() -> list:
    """bytes of lengths 0, 1, 4, 11, 12, 13, 16 and 70 KB; an embedded NUL; a 2-byte UTF-8 character across byte 12"""
    return [b"", b"a", b"abcd", b"hello world", b"twelve bytes", b"thirteen byte", b"sixteen bytes!!!", (bytes(range(32, 127)) * (BIG // 95 + 1))[:BIG],
            b"nul\x00inside", b"\x00" * 13, b"abcdefghijk\xc3\xa9xyz", "élan 😀".encode()]


DECIMAL_WIDTHS = [1, 4, 5, 9, 10, 18, 19, 38]


def _decimal_pairs() -> list:
    """(Arrow precision, table width, scale): every width at its own precision, and precisions below the width that
    cross each narrowing class"""
    out = []
    for w in DECIMAL_WIDTHS:
        for p in sorted({w, 1, 4, 9, 18} & set(range(1, w + 1))):
            out.append((p, w, min(p, 2)))
    return out


def accepted_pairs() -> list:
    """(id, Arrow type, column type, table DECIMAL (w, s) or None, edge values as Python values or raw bits)"""
    out = [("bool", pa.bool_(), ch.T_BOOLEAN, None, [True, False])]
    for bits, signed, t in ((8, True, ch.T_TINYINT), (8, False, ch.T_UTINYINT), (16, True, ch.T_SMALLINT), (16, False, ch.T_USMALLINT),
                            (32, True, ch.T_INTEGER), (32, False, ch.T_UINTEGER), (64, True, ch.T_BIGINT), (64, False, ch.T_UBIGINT)):
        typ = getattr(pa, ("int" if signed else "uint") + str(bits))()
        out.append((f"{typ}", typ, t, None, _int_edges(bits, signed)))
    out.append(("uint64-time_tz", pa.uint64(), ch.T_TIME_TZ, None, _int_edges(64, False)))
    out.append(("float32", pa.float32(), ch.T_FLOAT, None, F32_BITS))
    out.append(("float64", pa.float64(), ch.T_DOUBLE, None, F64_BITS))
    out.append(("date32", pa.date32(), ch.T_DATE, None, DATE_EDGES))
    out.append(("time64us", pa.time64("us"), ch.T_TIME, None, TIME_EDGES["us"]))
    out.append(("time64ns", pa.time64("ns"), ch.T_TIME_NS, None, TIME_EDGES["ns"]))
    for unit, t in (("s", ch.T_TIMESTAMP_S), ("ms", ch.T_TIMESTAMP_MS), ("us", ch.T_TIMESTAMP), ("ns", ch.T_TIMESTAMP_NS)):
        out.append((f"ts_{unit}", pa.timestamp(unit), t, None, _ts_edges(unit)))
    out.append(("ts_us_utc", pa.timestamp("us", tz="UTC"), ch.T_TIMESTAMP_TZ, None, _ts_edges("us")))
    out.append(("ts_us-tz_col", pa.timestamp("us"), ch.T_TIMESTAMP_TZ, None, _ts_edges("us")))
    for p, w, s in _decimal_pairs():
        out.append((f"d{p},{s}-DECIMAL({w},{s})", pa.decimal128(p, s), ch.T_DECIMAL, (w, s), decimal_values(p, s)))
    for p in (38, 20, 1):
        out.append((f"d{p},0-HUGEINT", pa.decimal128(p, 0), ch.T_HUGEINT, None, decimal_values(p, 0)))
    uhuge = [(2**128 - 1).to_bytes(16, "little"), bytes(16), (1).to_bytes(16, "little"), (2**127).to_bytes(16, "little"), bytes(range(16))]
    out.append(("fsb16-UHUGEINT", pa.binary(16), ch.T_UHUGEINT, None, uhuge))
    out.append(("fsb16-UUID", pa.binary(16), ch.T_UUID, None, uhuge))
    for typ, t in ((pa.string(), ch.T_VARCHAR), (pa.large_string(), ch.T_VARCHAR), (pa.binary(), ch.T_BLOB), (pa.large_binary(), ch.T_BLOB)):
        out.append((f"{typ}", typ, t, None, string_edges()))
    return out


PAIRS = accepted_pairs()
PAIR_IDS = [p[0] for p in PAIRS]


# ---------------------------------------------------------------------------------------------- building columns
def _fixed_payload(typ, values) -> bytes:
    """the raw Arrow value bytes of `values` (float edges are bit patterns)"""
    if pa.types.is_boolean(typ):
        return bytes(np.packbits(np.asarray(values, dtype=bool), bitorder="little"))
    if pa.types.is_floating(typ):
        return struct.pack(f"<{len(values)}{'I' if typ.bit_width == 32 else 'Q'}", *values)
    if pa.types.is_fixed_size_binary(typ):
        return b"".join(values)
    if pa.types.is_decimal(typ):
        return b"".join(rs.unscaled(v, typ.scale).to_bytes(16, "little", signed=True) for v in values)
    fmt = {8: "b", 16: "h", 32: "i", 64: "q"}[typ.bit_width]
    if pa.types.is_unsigned_integer(typ):
        fmt = fmt.upper()
    return struct.pack(f"<{len(values)}{fmt}", *values)


def _bitmap(valid) -> "pa.Buffer":
    return pa.py_buffer(np.packbits(np.asarray(valid, dtype=bool), bitorder="little").tobytes())


def column(typ, edges: list, idx, valid) -> "pa.Array":
    """Arrow array whose row r holds edges[idx[r]], NULL where not valid[r] over that payload (never zeroed).  String
    data buffers are sized exactly: the last row's bytes end at the buffer's last byte."""
    n = len(idx)
    bm = _bitmap(valid)
    nulls = int(n - np.count_nonzero(valid))
    if pa.types.is_string(typ) or pa.types.is_large_string(typ) or pa.types.is_binary(typ) or pa.types.is_large_binary(typ):
        strs = [edges[i] for i in idx]
        offs = np.zeros(n + 1, dtype=np.int64 if typ in (pa.large_string(), pa.large_binary()) else np.int32)
        np.cumsum([len(s) for s in strs], out=offs[1:])
        return pa.Array.from_buffers(typ, n, [bm, pa.py_buffer(offs.tobytes()), pa.py_buffer(b"".join(strs))], null_count=nulls)
    if pa.types.is_boolean(typ):
        payload = _fixed_payload(typ, [edges[i] for i in idx])
    else:
        one = _fixed_payload(typ, edges)
        w = len(one) // len(edges)
        payload = b"".join(one[i * w:(i + 1) * w] for i in idx)
    return pa.Array.from_buffers(typ, n, [bm, pa.py_buffer(payload)], null_count=nulls)


# ---------------------------------------------------------------------------------------------- placement
SUB_ROWS = 4096             # DMB_REV_BATCH_ROWS of the GPU tests: sub-batches of two chunks
APPEND_ROWS = 4096 + 2049   # rows per append: sub-batches [0, 4096) and [4096, 6145); chunk 3 is one row
NCOLS = 8                   # columns of one table; column c's child array starts at Arrow offset c + STRUCT_SLICE
STRUCT_SLICE = 3


def stride_for(e: int) -> int:
    """a stride coprime with the edge count (and odd, so coprime with the 2048-row chunks too when e is odd)"""
    s = 7
    while math.gcd(s, e) != 1:
        s += 2
    return s


def appends_for(e: int) -> int:
    """appends enough for every column shift 0 .. 2e-1: each edge twice at each row, once valid at least"""
    return (2 * e + NCOLS - 1) // NCOLS


def placement(e: int, j: int, c: int):
    """(edge index, valid) per row of append j, column c: edges on a stride coprime with e, shifted by j * NCOLS + c;
    every 4th run of e rows NULL, in a phase that moves when the shift wraps past e, so that a row NULL under one shift of an
    edge is valid under the next"""
    s = stride_for(e)
    r = np.arange(APPEND_ROWS)
    shift = j * NCOLS + c
    idx = (r * s + shift) % e
    valid = (r // e + shift // e) % 4 != 3
    return idx, valid


def positions(w: int) -> dict:
    """the rows of one append that the reverse kernels treat specially, for a vector payload of w bytes"""
    pos = {"chunk row 0": [0, 2048, 4096, 6144], "chunk row 2047": [2047, 4095],
           "sub-batch first": [0, 4096], "sub-batch last": [4095, APPEND_ROWS - 1]}
    per_vec = 16 // w if w in (1, 2, 4, 8, 16) else 1
    tail = [r for r0, r1 in ((0, 4096), (4096, APPEND_ROWS)) for r in range(r1 - (r1 - r0) % per_vec, r1)]
    if tail:
        pos["rev_copy tail"] = tail
    return pos


def struct_for(typ, edges: list, j: int) -> "pa.StructArray":
    """append j's batch: NCOLS columns, column c sliced from an array c rows longer, the struct sliced by STRUCT_SLICE"""
    e = len(edges)
    kids = []
    for c in range(NCOLS):
        idx, valid = placement(e, j, c)
        lead = c + STRUCT_SLICE
        full = column(typ, edges, np.concatenate([np.zeros(lead, np.int64), idx]), np.concatenate([np.ones(lead, bool), valid]))
        kids.append(full.slice(c))
    return pa.StructArray.from_arrays(kids, names=[f"c{c}" for c in range(NCOLS)]).slice(STRUCT_SLICE)


@pytest.mark.parametrize("w", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("e", [2, 7, 8, 9, 12, 13])
def test_placement_puts_every_edge_at_every_position(w, e):
    for name, rows in positions(w).items():
        seen = set()
        for j in range(appends_for(e)):
            for c in range(NCOLS):
                idx, valid = placement(e, j, c)
                seen |= {int(idx[r]) for r in rows if valid[r]}
        assert seen == set(range(e)), (name, sorted(set(range(e)) - seen))
    for c in range(NCOLS):  # every column (every Arrow offset) holds every edge, valid and NULL
        idx, valid = placement(e, 0, c)
        assert set(idx[valid].tolist()) == set(range(e)) and (~valid).any()


def test_placement_crosses_the_positions_of_a_real_batch():
    typ = pa.int16()
    edges = _int_edges(16, True)
    struct = struct_for(typ, edges, 1)
    assert len(struct) == APPEND_ROWS
    assert sorted({struct.field(c).offset % 8 for c in range(NCOLS)}) == list(range(8))
    for c in range(NCOLS):
        idx, valid = placement(len(edges), 1, c)
        assert struct.field(c).to_pylist() == [edges[i] if v else None for i, v in zip(idx, valid)]


# ---------------------------------------------------------------------------------------------- known answers
def test_known_decimal_and_integer_cells():
    arr = pa.array([Decimal("-12.3"), None, Decimal("999.9")], pa.decimal128(4, 1))
    assert rs.expected_cells(arr, ch.T_DECIMAL, (4, 1)) == [-123, None, 9999]
    assert rs.decode_cell(bytes.fromhex("85ff"), ch.T_DECIMAL) == -123
    assert rs.vector_width(ch.T_DECIMAL, 4) == 2 and rs.vector_width(ch.T_DECIMAL, 5) == 4
    assert rs.vector_width(ch.T_DECIMAL, 18) == 8 and rs.vector_width(ch.T_DECIMAL, 19) == 16
    # a narrower Arrow precision takes the table's scale and width: 1.5 in DECIMAL(18,2) is the int64 150
    arr = pa.array([Decimal("1.5"), Decimal("-12.25")]).cast(pa.decimal128(4, 2))
    assert rs.expected_cells(arr, ch.T_DECIMAL, (18, 2)) == [150, -1225]
    assert rs.decode_vector((150).to_bytes(8, "little", signed=True) + (-1225).to_bytes(8, "little", signed=True), None, 2,
                            ch.T_DECIMAL, 18) == [150, -1225]
    big = pa.array([Decimal(10**38 - 1), Decimal(-(10**38 - 1))], pa.decimal128(38, 0))
    assert rs.expected_cells(big, ch.T_HUGEINT) == [10**38 - 1, -(10**38 - 1)]
    assert rs.decode_cell((-(10**38 - 1)).to_bytes(16, "little", signed=True), ch.T_HUGEINT) == -(10**38 - 1)
    assert rs.decode_cell(b"\xff" * 8, ch.T_UBIGINT) == 2**64 - 1 and rs.decode_cell(b"\xff" * 8, ch.T_BIGINT) == -1


def test_known_temporal_and_float_cells():
    d = pa.array([rs.I32_MAX, -rs.I32_MAX, 0, -719162], pa.int32()).cast(pa.date32())
    assert rs.expected_cells(d, ch.T_DATE) == [rs.I32_MAX, -rs.I32_MAX, 0, -719162]
    ts = pa.array([I64_MAX, -I64_MAX, 1_000_000, None], pa.int64()).cast(pa.timestamp("us"))
    assert rs.expected_cells(ts, ch.T_TIMESTAMP) == [I64_MAX, -I64_MAX, 1_000_000, None]
    assert rs.expected_cells(pa.array([86_400_000_000], pa.int64()).cast(pa.time64("us")), ch.T_TIME) == [86_400_000_000]
    s = pa.array([-62135596800], pa.int64()).cast(pa.timestamp("s"))
    assert rs.expected_cells(s, ch.T_TIMESTAMP_S) == [-62135596800]
    f = pa.Array.from_buffers(pa.float32(), 2, [None, pa.py_buffer(struct.pack("<2I", 0x7FA00005, 0x80000000))])
    assert rs.expected_cells(f, ch.T_FLOAT) == [0x7FA00005, 0x80000000]  # the signalling NaN keeps its bits
    assert rs.expected_cells(pa.array([True, None, False]), ch.T_BOOLEAN) == [1, None, 0]


def test_known_string_cells():
    hello = bytes.fromhex("0500000068656c6c6f") + bytes(7)
    assert rs.decode_cell(hello, ch.T_VARCHAR) == b"hello"
    long = b"thirteen byte"
    keep = ctypes.create_string_buffer(long, len(long))
    e = struct.pack("<I", 13) + long[:4] + struct.pack("<Q", ctypes.addressof(keep))
    assert rs.decode_cell(e, ch.T_BLOB) == long
    with pytest.raises(AssertionError, match="prefix"):
        rs.decode_cell(struct.pack("<I", 13) + b"xxxx" + struct.pack("<Q", ctypes.addressof(keep)), ch.T_VARCHAR)
    with pytest.raises(AssertionError, match="padding"):
        rs.decode_cell(hello[:-1] + b"\x01", ch.T_VARCHAR)
    assert rs.expected_cells(pa.array(["é", None, "a\x00b"]), ch.T_VARCHAR) == ["é".encode(), None, b"a\x00b"]


def test_decoder_holds_the_vector_invariants():
    valid = np.zeros(32, np.uint64)
    valid[0] = 0b101
    vb = valid.tobytes()
    assert rs.decode_vector(struct.pack("<3i", 7, 0, -7), vb, 3, ch.T_INTEGER) == [7, None, -7]
    with pytest.raises(AssertionError, match="NULL payload"):
        rs.decode_vector(struct.pack("<3i", 7, 1, -7), vb, 3, ch.T_INTEGER)
    assert rs.decode_vector(struct.pack("<3i", 7, 1, -7), vb, 3, ch.T_INTEGER, strict=False) == [7, None, -7]
    past = valid.copy()
    past[0] |= 1 << 3
    with pytest.raises(AssertionError, match="past count"):
        rs.decode_vector(struct.pack("<3i", 7, 0, -7), past.tobytes(), 3, ch.T_INTEGER)
    with pytest.raises(AssertionError, match="BOOLEAN"):
        rs.decode_vector(bytes([1, 0, 2]), None, 3, ch.T_BOOLEAN)
    lvalid = np.zeros(32, np.uint64)
    lvalid[0] = 0b101
    child = struct.pack("<2h", 3, -4)
    ent = struct.pack("<6Q", 0, 2, 2, 0, 2, 0)
    assert rs.decode_list_vector(ent, lvalid.tobytes(), 3, child, None, 2, ch.T_SMALLINT) == [[3, -4], None, []]
    with pytest.raises(AssertionError, match="NULL list"):  # a NULL row keeps length 0 whatever Arrow gave it
        rs.decode_list_vector(struct.pack("<6Q", 0, 2, 1, 1, 2, 0), lvalid.tobytes(), 3, child, None, 2, ch.T_SMALLINT)
    with pytest.raises(AssertionError, match="leaves the child"):
        rs.decode_list_vector(struct.pack("<6Q", 0, 3, 2, 0, 2, 0), lvalid.tobytes(), 3, child, None, 2, ch.T_SMALLINT)


@pytest.mark.parametrize("precision,scale,bits,type_id,table,why", [
    (9, 2, 32, ch.T_DECIMAL, (9, 2), "32-bit"), (18, 2, 64, ch.T_DECIMAL, (18, 2), "64-bit"), (40, 2, 256, ch.T_DECIMAL, None, "256-bit"),
    (18, 3, 128, ch.T_DECIMAL, (18, 2), "scale"), (38, 2, 128, ch.T_DECIMAL, (18, 2), "precision"), (20, 4, 128, ch.T_HUGEINT, None, "scale"),
    (4, 2, 128, ch.T_DECIMAL, (18, 2), None), (38, 0, 128, ch.T_HUGEINT, None, None), (5, 1, 128, ch.T_DECIMAL, None, None)])
def test_decimal_refusals(precision, scale, bits, type_id, table, why):
    assert rs.decimal_refusal(precision, scale, bits, type_id, table) == why


# ---------------------------------------------------------------------------------------------- the oracle
def table_op(type_id: int, dec_width: int) -> int:
    """the DMB_REV_* op a column of this table type implies (DECIMAL: by the table's width)"""
    if type_id == ch.T_BOOLEAN:
        return 5
    if type_id == ch.T_DECIMAL:
        return {2: 8, 4: 7, 8: 6, 16: 4}[rs.decimal_width_bytes(dec_width)]
    return {1: 0, 2: 1, 4: 2, 8: 3, 16: 4}[rs.vector_width(type_id)]


def _oracle_vectors(arr, type_id, dec_width):
    import oracle
    n, off = len(arr), arr.offset
    bufs = arr.buffers()
    bitmap = np.frombuffer(bufs[0], dtype=np.uint8) if bufs[0] is not None else None
    if type_id in rs.STRINGS:
        ow = 8 if arr.type in (pa.large_string(), pa.large_binary()) else 4
        offsets = np.frombuffer(bufs[1], dtype=np.int64 if ow == 8 else np.int32)[off:off + n + 1].copy()
        data = np.frombuffer(bufs[2], dtype=np.uint8)
        return oracle.rev_string(offsets, data, bufs[2].address, bitmap, off, n)[:2], 16
    if type_id == ch.T_BOOLEAN:
        return oracle.rev_fixed(np.frombuffer(bufs[1], dtype=np.uint8), bitmap, off, n, 5, 1)[:2], 1
    w_in = 16 if pa.types.is_decimal(arr.type) else arr.type.bit_width // 8
    vals = np.frombuffer(bufs[1], dtype=np.uint8)[off * w_in:].copy()
    w_out = rs.vector_width(type_id, dec_width)
    return oracle.rev_fixed(vals, bitmap, off, n, table_op(type_id, dec_width), w_out)[:2], w_out


@pytest.mark.parametrize("pair", PAIRS, ids=PAIR_IDS)
def test_oracle_reverse_conversions_match_the_reference(pair):
    _, typ, type_id, table, edges = pair
    dec_width = table[0] if table else 0
    struct_arr = struct_for(typ, edges, 0)
    for c in (0, 5):
        arr = struct_arr.field(c)
        (out, val), w = _oracle_vectors(arr, type_id, dec_width)
        got = []
        for k in range((len(arr) + 2047) // 2048):
            cnt = min(2048, len(arr) - 2048 * k)
            got += rs.decode_vector(out[k * 2048 * w:(k * 2048 + cnt) * w].tobytes(), val[32 * k:32 * k + 32].tobytes(), cnt, type_id, dec_width)
        assert got == rs.expected_cells(arr, type_id, table)
