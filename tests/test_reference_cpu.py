"""The CPU oracle against tests/reference_semantics.py, on the values where DuckDB's casts and renderings differ from the
easy cases: ties, +-2^63, NaN / inf / -0.0, subnormals, the 1e-5 / 1e16 layout boundaries, every integer width's
limits, the 128-bit renderer's limb boundaries, DECIMAL ties at every storage width, calendar edges, BC and 5-digit
years and DuckDB's infinite DATE / TIMESTAMP.  No GPU: tests/test_gpu_reference.py runs the same edge sets on the device.

An edge column is a list of values of one logical type, the getter casts that apply to it (dst kind -> reference
function) and its VARCHAR rendering.  Batches place edge value `(q k + r) % E` at row r of chunk k, q the smallest prime that does not divide E, so with enough
chunks every value is seen at row 0, inside the 16-byte vectors and in a chunk's scalar tail."""
import datetime
import math
import struct

import numpy as np
import pytest

import oracle
import reference_semantics as rs
from duckdb_mbt_b200 import chunks as ch


def f64_bits(b: int) -> float:
    return struct.unpack("<d", struct.pack("<Q", b))[0]


def next_toward_zero(v: float) -> float:
    return math.nextafter(v, 0.0)


def f32(v) -> float:
    return float(np.float32(v))


def f32_next(v, toward) -> float:
    return float(np.nextafter(np.float32(v), np.float32(toward)))


def days_of(y, m, d) -> int:
    return datetime.date(y, m, d).toordinal() - datetime.date(1970, 1, 1).toordinal()


NEG_NAN = f64_bits(0xFFF8000000000000)

DOUBLES = [0.0, -0.0, 0.5, -0.5, 1.5, -1.5, 2.5, -2.5, 0.49999999999999994, 4503599627370495.5, -4503599627370495.5,
           2.0 ** 63, -(2.0 ** 63), next_toward_zero(2.0 ** 63), next_toward_zero(-(2.0 ** 63)),
           float("nan"), NEG_NAN, float("inf"), float("-inf"),
           5e-324, -5e-324, f64_bits(0x000FFFFFFFFFFFFF), 1.7976931348623157e308, -1.7976931348623157e308,
           1e-5, math.nextafter(1e-5, 0.0), math.nextafter(1e-5, 1.0), -1e-5,
           1e16, math.nextafter(1e16, 0.0), math.nextafter(1e16, 2e16), -1e16, 9999999999999998.0,
           0.1, 1.0 / 3.0, 123456.789, 2.0 ** 53 + 2.0, -(2.0 ** 31) - 0.5, 2.0 ** 31 - 0.5]

FLOATS = [f32(v) for v in [0.0, -0.0, 0.1, 1.1, -1.1, 0.5, 1.5, 2.5, -2.5, 8388607.5, 2.0 ** 24, f32(3.4028234663852886e38), -f32(3.4028234663852886e38),
          f32(1.401298464324817e-45), f32_next(1.1754943508222875e-38, 0), 1.1754943508222875e-38,
          2.0 ** 63, -(2.0 ** 63), f32_next(2.0 ** 63, 0), f32_next(-(2.0 ** 63), 0),
          f32(1e-5), f32_next(1e-5, 0), f32_next(1e-5, 1), f32(1e16), f32_next(1e16, 0), f32_next(1e16, 2e16),
          float("nan"), NEG_NAN, float("inf"), float("-inf"), 3.14159, 1e-10, 123456.79, 16777215.0]]

INT_LIMITS = {ch.T_TINYINT: (-2**7, 2**7 - 1), ch.T_SMALLINT: (-2**15, 2**15 - 1), ch.T_INTEGER: (-2**31, 2**31 - 1),
              ch.T_BIGINT: (-2**63, 2**63 - 1), ch.T_UTINYINT: (0, 2**8 - 1), ch.T_USMALLINT: (0, 2**16 - 1),
              ch.T_UINTEGER: (0, 2**32 - 1), ch.T_UBIGINT: (0, 2**64 - 1)}


def int_values(type_id):
    lo, hi = INT_LIMITS[type_id]
    vals = [lo, lo + 1, hi, hi - 1, 0, 1, -1, 2**31 - 1, -2**31, 2**31, 2**32 - 1, 2**53 + 1, 2**63 - 1, 2**63, 2**64 - 1]
    return sorted({v for v in vals if lo <= v <= hi}, key=lambda v: (abs(v), v))


HUGE_K = (18, 19, 20, 37, 38)
HUGEINTS = ([-2**127, 2**127 - 1, 0, 1, -1] + [s * v for k in HUGE_K for v in (10**k, 10**k - 1) for s in (1, -1)]
            + [2**63 - 1, 2**63, 2**64 - 1, 2**64, -2**63, -2**63 - 1, -2**64, -2**64 + 1, 2**53 + 1, -(2**53) - 1])
UHUGEINTS = ([0, 1, 2**128 - 1, 2**127] + [v for k in HUGE_K for v in (10**k, 10**k - 1)]
             + [2**63 - 1, 2**63, 2**64 - 1, 2**64, 2**53 + 1])


def decimal_values(width, scale):
    p, top = 10 ** scale, 10 ** width - 1
    vals = {0, 1, -1, top, -top}
    if scale < width:
        vals |= {p, -p}
    if scale >= 1:
        for t in (p // 2, 3 * p // 2, top // p * p + p // 2 if top // p * p + p // 2 <= top else p // 2):
            vals |= {t, -t, t - 1, -(t - 1)}
    if width >= 16:
        vals |= {2**53, -(2**53), 2**53 + 1, -(2**53) - 1}
    if width == 38:  # rounded results that leave int64
        for q in (2**63 - 1, 2**63, -(2**63), -(2**63) - 1):
            vals |= {q * p, q * p + (p // 2 if q >= 0 else -(p // 2)), q * p + (p // 2 - 1 if q >= 0 else -(p // 2 - 1))}
    return sorted((v for v in vals if abs(v) <= top), key=lambda v: (abs(v), v))  # DECIMAL(w, s) holds |x| < 10^w


DATES = [0, 1, -1, days_of(1900, 2, 28), days_of(1900, 3, 1), days_of(2000, 2, 29), days_of(2100, 2, 28), days_of(2100, 3, 1),
         days_of(1, 1, 1), days_of(1, 1, 1) - 1, days_of(9999, 12, 31), days_of(9999, 12, 31) + 1, days_of(1968, 1, 1),
         days_of(1969, 12, 31), days_of(1600, 2, 29), days_of(1582, 10, 4), days_of(1, 1, 1) - 366 - 365,
         2**31 - 1, -(2**31 - 1), 2**31 - 2, -(2**31 - 2)]
US = 1_000_000
TS_MIN_US = -9223372022400000000  # 290309-12-22 (BC) 00:00:00, DuckDB's lowest finite TIMESTAMP
TIMESTAMPS = [0, 1, -1, -US + 1, -US, -US - 1, 86400 * US - 1, days_of(1, 1, 1) * 86400 * US - 1, 2**63 - 2, TS_MIN_US,
              days_of(2000, 2, 29) * 86400 * US + 43200 * US + 123456, 2**63 - 1, -(2**63 - 1)]
TS_S = [0, 1, -1, 9223372036854, TS_MIN_US // US, days_of(1, 1, 1) * 86400 - 1, 86399]
TS_MS = [0, 1, -1, -999, -1000, -1001, 9223372036854775, TS_MIN_US // 1000, 1500, 10]
TS_NS = [0, 1, -1, -999, -1000, -1001, 999, 2**63 - 2, -(2**63) + 2, 1_000_000_000, 123_000_000, 10]
TIMES = [0, 1, 86399999999, 86400 * US, 12 * 3600 * US + 500000, 59 * US + 10]
TIMES_NS = [0, 1, 999, 86400 * 10**9 - 1, 86400 * 10**9, 1000]
UUIDS = [0, 2**128 - 1, 2**127, 2**127 - 1, 0x0123456789ABCDEF0123456789ABCDEF, 1]
# INTERVAL (months, days, micros): month_day_nano keeps months and days and scales micros where nanoseconds fit int64
INTERVALS = [(0, 0, 0), (1, 1, 1), (-1, -1, -1), (2**31 - 1, 2**31 - 1, rs.I64_MAX // 1000), (-(2**31), -(2**31), -(rs.I64_MAX // 1000)),
             (12, 30, 86400 * US), (0, 0, -999), (-13, 400, 123456789)]


def _i64_casts(to_int, to_f64=float):
    return {ch.D_I64: lambda x: rs.int_to_i64(to_int(x)), ch.D_I32_TRUNC: lambda x: rs.i32_trunc(rs.int_to_i64(to_int(x))),
            ch.D_F64: to_f64, ch.D_BOOL_BYTE: rs.bool_byte}


def _float_casts():
    return {ch.D_I64: rs.to_i64, ch.D_I32_TRUNC: lambda v: rs.i32_trunc(rs.to_i64(v)), ch.D_F64: lambda v: v,
            ch.D_BOOL_BYTE: rs.bool_byte}


def dec_bool_pinned(x, s):
    """DECIMAL -> BOOLEAN is the rounded integer != 0; where that integer leaves int64 (width 38 only) the getter's
    answer is UNPINNED (DESIGN.md section 1) and the value is left out (None)"""
    q = rs.dec_round(x, s)
    return int(q != 0) if rs.fits_i64(q) else None


def month_day_nano(iv):
    months, days, micros = iv
    return int.from_bytes(struct.pack("<iiq", months, days, rs.month_day_nano(micros)), "little")


def edge_columns():
    """[(name, type_id, dec_width, dec_scale, values, {dst: reference}, render or None)]"""
    cols = [("bool", ch.T_BOOLEAN, 0, 0, [0, 1], _i64_casts(lambda x: x), lambda v: "true" if v else "false"),
            ("f64", ch.T_DOUBLE, 0, 0, DOUBLES, _float_casts(), rs.render_double),
            ("f32", ch.T_FLOAT, 0, 0, FLOATS, _float_casts(), rs.render_float)]
    for t in INT_LIMITS:
        casts = _i64_casts(lambda x: x)
        casts[ch.D_I32_SAT] = rs.i32_sat
        if t == ch.T_BIGINT:
            casts[ch.D_I128] = lambda x: x
        cols.append((f"int{t}", t, 0, 0, int_values(t), casts, rs.render_int))
    huge = _i64_casts(lambda x: x, rs.huge_to_f64)
    huge[ch.D_I128] = lambda x: x
    cols.append(("huge", ch.T_HUGEINT, 0, 0, HUGEINTS, huge, rs.render_int))
    cols.append(("uhuge", ch.T_UHUGEINT, 0, 0, UHUGEINTS, _i64_casts(lambda x: x, rs.uhuge_to_f64), rs.render_int))
    for w in (4, 9, 18, 38):
        for s in sorted({0, 1, w - 1, w}):
            casts = {ch.D_DEC_I64: lambda x, s=s: rs.dec_to_i64(x, s),
                     ch.D_DEC_I32_TRUNC: lambda x, s=s: rs.i32_trunc(rs.dec_to_i64(x, s)),
                     ch.D_DEC_F64: lambda x, s=s, w=w: rs.dec_to_f64(x, s, w),
                     ch.D_DEC_BOOL_BYTE: lambda x, s=s: dec_bool_pinned(x, s), ch.D_I128: lambda x: x}
            cols.append((f"dec{w}_{s}", ch.T_DECIMAL, w, s, decimal_values(w, s), casts, lambda x, s=s: rs.render_decimal(x, s)))
    cols += [("date", ch.T_DATE, 0, 0, DATES, {ch.D_DATE_REF: rs.date_ref}, rs.render_date),
             ("ts", ch.T_TIMESTAMP, 0, 0, TIMESTAMPS, {}, rs.render_timestamp),
             ("ts_tz", ch.T_TIMESTAMP_TZ, 0, 0, TIMESTAMPS, {}, lambda v: rs.render_timestamp(v, tz=True)),
             ("ts_s", ch.T_TIMESTAMP_S, 0, 0, TS_S, {ch.D_TS_US_FROM_S: rs.ts_us_from_s}, lambda v: rs.render_timestamp(v, "s")),
             ("ts_ms", ch.T_TIMESTAMP_MS, 0, 0, TS_MS, {ch.D_TS_US_FROM_MS: rs.ts_us_from_ms}, lambda v: rs.render_timestamp(v, "ms")),
             ("ts_ns", ch.T_TIMESTAMP_NS, 0, 0, TS_NS, {ch.D_TS_US_FROM_NS: rs.ts_us_from_ns}, lambda v: rs.render_timestamp(v, "ns")),
             ("time", ch.T_TIME, 0, 0, TIMES, {}, rs.render_time),
             ("time_ns", ch.T_TIME_NS, 0, 0, TIMES_NS, {}, lambda v: rs.render_time(v, "ns")),
             ("uuid", ch.T_UUID, 0, 0, UUIDS, {}, rs.render_uuid),
             ("interval", ch.T_INTERVAL, 0, 0, INTERVALS, {ch.D_MONTH_DAY_NANO: month_day_nano}, None)]
    for col in cols:  # the raw copy, NULL slots zeroed: what every fixed-width Arrow column starts from
        col[5][ch.D_SAME] = None
    return cols


EDGE_COLUMNS = edge_columns()
WIDTH_OF_DST = {ch.D_I64: 8, ch.D_I32_TRUNC: 4, ch.D_F64: 8, ch.D_BOOL_BYTE: 1, ch.D_I128: 16, ch.D_I32_SAT: 4,
                ch.D_TS_US_FROM_S: 8, ch.D_TS_US_FROM_MS: 8, ch.D_TS_US_FROM_NS: 8, ch.D_DATE_REF: 4,
                ch.D_DEC_I64: 8, ch.D_DEC_I32_TRUNC: 4, ch.D_DEC_F64: 8, ch.D_DEC_BOOL_BYTE: 1, ch.D_MONTH_DAY_NANO: 16}


def out_width(col, dst) -> int:
    return ch.PHYS_WIDTH[ch.phys_of_type(col[1], col[2])] if dst == ch.D_SAME else WIDTH_OF_DST[dst]


def text_pinned(type_id, v) -> bool:
    """inputs whose text is UNPINNED (DESIGN.md section 1) stay out of the text checks: a NaN with the sign bit set"""
    return not (type_id in (ch.T_DOUBLE, ch.T_FLOAT) and math.isnan(v) and math.copysign(1.0, v) < 0)


# ---------------------------------------------------------------- batches
def payload(type_id, dec_width, values) -> np.ndarray:
    phys = ch.phys_of_type(type_id, dec_width)
    if type_id == ch.T_INTERVAL:
        return np.stack([np.frombuffer(struct.pack("<iiq", *v), np.uint8) for v in values])
    if ch.PHYS_WIDTH[phys] == 16:
        return np.stack([np.frombuffer((v & (2**128 - 1)).to_bytes(16, "little"), np.uint8) for v in values])
    if phys == ch.P_F32:
        return np.asarray(values, dtype=np.float64).astype(np.float32)  # NaN payloads: the sign survives
    if phys == ch.P_F64:
        return np.asarray(values, dtype=np.float64)
    dt = ch.PHYS_NUMPY[phys]
    return np.asarray([v & ((1 << (8 * np.dtype(dt).itemsize)) - 1) for v in values], dtype=np.uint64).astype(dt) \
        if np.dtype(dt).kind == "u" else np.asarray(values, dtype=dt)


def chunk_stride(e: int) -> int:
    """the smallest prime that does not divide e: k -> stride * k % e then visits every edge value"""
    return next(q for q in (2, 3, 5, 7, 11, 13, 17, 19, 23, 29) if e % q)


def placement(counts: np.ndarray, e: int) -> np.ndarray:
    """edge index of every row: value (q k + r) % e at row r of chunk k, q = chunk_stride(e)"""
    q = chunk_stride(e)
    parts = [(q * k + np.arange(int(c))) % e for k, c in enumerate(counts)]
    return np.concatenate(parts).astype(np.int64) if parts else np.zeros(0, np.int64)


def position_counts(e: int) -> np.ndarray:
    """2e chunks alternating 2033 and 2047 rows: 2033 = 1 mod 16 and 2047 = 15 mod 16 leave a scalar tail for every
    rows-per-vector R in {2, 4, 8, 16}; with placement()'s stride the chunks' rows 0 and their tail rows take every
    edge value (test_positions_cover_every_edge_value)"""
    return np.asarray([2033 if k % 2 == 0 else 2047 for k in range(2 * e)], dtype=np.uint32)


def edge_batch(cols, counts, rng=None, null_every=0):
    """cols: entries of EDGE_COLUMNS.  Returns (batch, [edge index per row], valid or None); NULL rows hold garbage."""
    n = int(counts.sum())
    valid = None
    if null_every:
        valid = (np.arange(n) % null_every) != null_every - 1
    cols_out, idxs = [], []
    for name, t, w, s, values, _, _ in cols:
        idx = placement(counts, len(values))
        pay = payload(t, w, values)[idx]
        cols_out.append(ch.fixed_column(name, t, pay, counts, valid=valid, dec_width=w, dec_scale=s,
                                        garbage_rng=rng if valid is not None else None))
        idxs.append(idx)
    return ch.ChunkBatch(counts, cols_out), idxs, valid


def expected_values(col, dst, idx, valid):
    """-> (uint8 [n, width] Arrow-layout output the reference function gives, NULL slots zero; bool [n] rows whose
    answer is pinned)"""
    name, t, w, s, values, casts, _ = col
    width = out_width(col, dst)
    n = idx.shape[0]
    if dst == ch.D_SAME:
        rows = np.ascontiguousarray(payload(t, w, values)).view(np.uint8).reshape(len(values), width)[idx].copy()
        known = np.ones(n, bool)
    else:
        table = [casts[dst](v) for v in values]
        known = np.asarray([x is not None for x in table])[idx]
        table = [0 if x is None else x for x in table]
        if dst in (ch.D_F64, ch.D_DEC_F64):
            rows = np.asarray(table, dtype=np.float64)[idx].view(np.uint8).reshape(n, 8).copy()
        elif width == 16:
            rows = np.stack([np.frombuffer((x & (2**128 - 1)).to_bytes(16, "little"), np.uint8) for x in table])[idx]
        else:
            dt = {8: np.int64, 4: np.int32, 1: np.uint8}[width]
            rows = np.asarray(table, dtype=dt)[idx].view(np.uint8).reshape(n, width).copy()
    if valid is not None:
        rows[~valid] = 0
        known = known | ~valid
    return rows, known


def value_mismatches(col, dst, got, idx, valid):
    """edge values whose output rows differ from the reference"""
    ev, known = expected_values(col, dst, idx, valid)
    got = got[: ev.size].reshape(ev.shape)
    rows = np.nonzero(known & (got != ev).any(axis=1))[0]
    return rows, sorted({str(col[4][idx[r]]) for r in rows[:50]})


TEXT_COLUMNS = [c for c in EDGE_COLUMNS if c[6] is not None]


def expected_texts(col, idx):
    name, t, w, s, values, _, render = col
    table = [render(v).encode() if text_pinned(t, v) else None for v in values]
    return [table[i] for i in idx]


# ---------------------------------------------------------------- the references themselves
def test_reference_semantics_known_answers():
    # FLOAT: the float's own digits; DOUBLE: repr's; the project's layout at 1e-5 / 1e16
    assert rs.render_float(f32(0.1)) == "0.1" and rs.render_float(f32(1.1)) == "1.1"
    assert rs.render_double(float(np.float32(0.1))) == "0.10000000149011612"
    assert rs.render_float(2.0 ** 24) == "16777216.0" and rs.render_float(f32(1e16)) == "1e+16"
    assert rs.render_float(f32(1.401298464324817e-45)) == "1e-45"
    assert rs.render_double(1e-5) == "0.00001" and rs.render_double(1e16) == "1e+16" and rs.render_double(-0.0) == "-0.0"
    assert rs.render_double(9999999999999998.0) == "9999999999999998.0" and rs.render_double(5e-324) == "5e-324"
    # casts
    assert [rs.to_i64(v) for v in (0.5, 1.5, 2.5, -2.5, 0.49999999999999994, 2.0 ** 63, -(2.0 ** 63))] == [0, 2, 2, -2, 0, 0, -2**63]
    assert rs.to_i64(4503599627370495.5) == 4503599627370496 and rs.to_i64(float("nan")) == 0
    assert rs.bool_byte(-0.0) == 0 and rs.bool_byte(float("nan")) == 1
    assert rs.ts_us_from_ns(-1) == -1 and rs.ts_us_from_ns(-1000) == -1 and rs.ts_us_from_ns(-1001) == -2
    assert rs.dec_to_i64(15, 1) == 2 and rs.dec_to_i64(-15, 1) == -2 and rs.dec_to_i64(14, 1) == 1 and rs.dec_to_i64(-25, 1) == -3
    assert rs.i32_trunc(2**31) == -2**31 and rs.i32_sat(2**40) == 2**31 - 1
    # SURVEY.md B.4: 1969-12-31 -> -1 is still right, 1968-01-01 loses 1968's leap day
    assert rs.date_to_days_ref(1969, 12, 31) == -1 and rs.date_to_days_ref(1970, 1, 1) == 0
    assert rs.date_to_days_ref(1968, 1, 1) == days_of(1968, 1, 1) + 1
    assert rs.date_ref(days_of(2024, 6, 3)) == 19877
    # calendar and infinities
    assert rs.render_date(days_of(1, 1, 1) - 1) == "0001-12-31 (BC)" and rs.render_date(days_of(9999, 12, 31) + 1) == "10000-01-01"
    assert rs.render_date(2**31 - 1) == "infinity" and rs.render_date(-(2**31 - 1)) == "-infinity"
    assert rs.render_date(2**31 - 2) == "5881580-07-10" and rs.render_date(-(2**31 - 2)) == "5877642-06-25 (BC)"
    assert rs.render_timestamp(-1) == "1969-12-31 23:59:59.999999" and rs.render_timestamp(-US + 1) == "1969-12-31 23:59:59.000001"
    assert rs.render_timestamp(2**63 - 1) == "infinity" and rs.render_timestamp(-(2**63 - 1), tz=True) == "-infinity"
    assert rs.render_timestamp(2**63 - 2) == "294247-01-10 04:00:54.775806"
    assert rs.render_timestamp(TS_MIN_US) == "290309-12-22 (BC) 00:00:00"
    assert rs.render_time(86400 * US) == "24:00:00" and rs.render_time(1, "ns") == "00:00:00.000000001"
    assert rs.render_uuid(2**127) == "00000000-0000-0000-0000-000000000000"
    assert rs.render_decimal(-5, 3) == "-0.005" and rs.render_decimal(10**38 - 1, 38) == "0." + "9" * 38


def test_reference_double_casts_stay_close_to_exact():
    # HUGEINT / UHUGEINT -> DOUBLE by DuckDB's formula is within one ulp of the correctly rounded conversion
    for x in HUGEINTS:
        assert rs.ulps_apart(rs.huge_to_f64(x), float(x)) <= 1, x
    for x in UHUGEINTS:
        assert rs.ulps_apart(rs.uhuge_to_f64(x), float(x)) <= 1, x
    # DECIMAL -> DOUBLE: bit exact where the division is exact-rounded, within 2 ulp of the exact quotient elsewhere
    for w in (4, 9, 18, 38):
        for s in sorted({0, 1, w - 1, w}):
            for x in decimal_values(w, s):
                got = rs.dec_to_f64(x, s, w)
                if abs(x) <= 2**53 and s <= 22:
                    assert got == rs.exact_f64(x, s), (w, s, x)
                else:
                    assert rs.ulps_apart(got, rs.exact_f64(x, s)) <= 2, (w, s, x)


# ---------------------------------------------------------------- the oracle
def _check_oracle(cols, counts, rng=None, null_every=0):
    batch, idxs, valid = edge_batch(cols, counts, rng, null_every)
    ora = oracle.OracleResult(batch)
    for j, col in enumerate(cols):
        name, t, w, s, values, casts, render = col
        for dst in casts:
            got, _, _, _ = ora.arrow_fixed(j, dst, out_width(col, dst))
            rows, bad = value_mismatches(col, dst, got, idxs[j], valid)
            if rows.size:
                pytest.fail(f"{name} dst={dst}: oracle differs from the reference for {bad[:8]}")
    return batch, idxs, valid, ora


@pytest.mark.parametrize("n,pattern", [(1, "full"), (2047, "full"), (2049, "full"), (6000, "ragged")])
def test_oracle_casts_match_the_references(n, pattern):
    rng = np.random.default_rng(70 + n)
    counts = ch.chunk_counts(n, pattern, rng)
    _check_oracle(EDGE_COLUMNS, counts, rng, null_every=7 if n > 1 else 0)


def test_positions_cover_every_edge_value():
    """position_counts + placement put every edge value at a chunk's row 0 and in a chunk's scalar tail (the last
    count % R rows) for every rows-per-vector R a conversion of the column can use"""
    for col in EDGE_COLUMNS:
        e = len(col[4])
        counts = position_counts(e)
        idx = placement(counts, e)
        starts = np.concatenate([[0], np.cumsum(counts[:-1], dtype=np.int64)])
        assert set(idx[starts].tolist()) == set(range(e)), col[0]
        w_in = ch.PHYS_WIDTH[ch.phys_of_type(col[1], col[2])]
        for r in (2, 4, 8, 16):
            if r * w_in > 16:
                continue
            tail = [i for k, c in enumerate(counts) for i in range(starts[k] + c - c % r, starts[k] + c)]
            assert set(idx[tail].tolist()) == set(range(e)), (col[0], r)


def test_oracle_casts_at_every_position():
    for col in EDGE_COLUMNS:
        _check_oracle([col], position_counts(len(col[4]))[:4])


@pytest.mark.parametrize("col", TEXT_COLUMNS, ids=[c[0] for c in TEXT_COLUMNS])
def test_oracle_text_matches_the_references(col):
    """duckdb_value_varchar of every edge value (cell_value) and the reference's string getter blob"""
    name, t, w, s, values, _, render = col
    counts = ch.chunk_counts(len(values))
    batch, idxs, _ = edge_batch([col], counts)
    ora = oracle.OracleResult(batch)
    exp = expected_texts(col, idxs[0])
    bad = [(values[idxs[0][i]], ora.cell_value(0, i), exp[i]) for i in range(len(exp)) if exp[i] is not None and ora.cell_value(0, i) != exp[i]]
    assert not bad, f"{name}: (value, oracle, reference) {bad[:6]}"
    keep = [i for i in range(len(exp)) if exp[i] is not None]
    if len(keep) == len(exp):
        stream = b"".join(x + b"\0" for x in exp)
        head = np.asarray([len(exp), len(stream)], dtype="<i4").tobytes()
        assert ora.get_column("string", 0) == head + stream
        assert ora.get_column("string", 0, nullable=True) == head + stream + b"\x01" * len(exp)


def test_oracle_float_text_matches_numpy_on_a_bit_pattern_sweep():
    """every 2^14-th float32 bit pattern plus every float of short runs around 1e-5, 1, 2^24 and 1e16 and a stride of
    subnormals: the oracle's float-shortest digits are numpy's"""
    pats = [np.arange(0, 2**32, 2**14, dtype=np.uint64).astype(np.uint32)]
    for v in (1e-5, 1.0, 2.0 ** 24, 1e16):
        b = int(np.float32(v).view(np.uint32))
        pats.append(np.arange(b - 600, b + 600, dtype=np.uint32))
    pats.append(np.arange(1, 2**23, 4099, dtype=np.uint32))
    bits = np.concatenate(pats)
    vals = bits.view(np.float32)
    keep = ~(np.isnan(vals) & np.signbit(vals))
    vals = vals[keep]
    counts = ch.chunk_counts(vals.shape[0])
    ora = oracle.OracleResult(ch.ChunkBatch(counts, [ch.fixed_column("f", ch.T_FLOAT, vals, counts)]))
    blob = ora.get_column("string", 0)
    got = blob[8:].split(b"\0")[: vals.shape[0]]
    bad = [(float(vals[i]), got[i]) for i in range(vals.shape[0]) if got[i] != rs.render_float(float(vals[i])).encode()]
    assert not bad, bad[:8]


def test_oracle_date_and_timestamp_text_on_random_days():
    rng = np.random.default_rng(3)
    days = rng.integers(-(2**31) + 2, 2**31 - 1, 2000).astype(np.int64)
    days[:1000] = rng.integers(-800_000, 3_000_000, 1000)
    micros = rng.integers(TS_MIN_US, 2**63 - 1, 2000, dtype=np.int64)
    counts = ch.chunk_counts(2000)
    ora = oracle.OracleResult(ch.ChunkBatch(counts, [ch.fixed_column("d", ch.T_DATE, days.astype(np.int32), counts),
                                                     ch.fixed_column("t", ch.T_TIMESTAMP, micros, counts)]))
    for i in range(2000):
        assert ora.cell_value(0, i).decode() == rs.render_date(int(days[i])), int(days[i])
        assert ora.cell_value(1, i).decode() == rs.render_timestamp(int(micros[i])), int(micros[i])
