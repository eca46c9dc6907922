"""Plain-Python statements of DuckDB's casts and VARCHAR renderings, independent of oracle/oracle.c and of the kernels.

Every function takes Python ints / floats and returns the expected value or text, computed with exact arithmetic
(`int`, `fractions.Fraction`, `datetime`, `uuid`, Python's and numpy's shortest float reprs).  Nothing here imports
torch or the oracle: the tests hold the oracle and the device to these functions, so a mistake shared by oracle.c and
the CUDA code shows up as a mismatch with a third, differently written statement.

The cast rules are those of the reference's getters (`duckdb_value_int64` / `_double` / `_boolean` cast the cell by its
logical type; a failed cast gives 0).  The renderings are DuckDB's VARCHAR casts.  The fixed / exponent layout of
DOUBLE and FLOAT text beyond the reference's fixture strings is the project's own rule, written once in `_layout`.
"""
from __future__ import annotations

import datetime
import functools
import math
import uuid
from decimal import Decimal
from fractions import Fraction

import numpy as np

I32_MIN, I32_MAX = -2**31, 2**31 - 1
I64_MIN, I64_MAX = -2**63, 2**63 - 1
U64_MAX = 2**64 - 1
TWO64 = 2.0 ** 64


# ---------------------------------------------------------------- integer casts
def fits_i64(x: int) -> bool:
    return I64_MIN <= x <= I64_MAX


def to_i64(v: float) -> int:
    """DOUBLE / FLOAT -> BIGINT: round half to even; NaN, +-inf and anything outside [-2^63, 2^63) fail (0)."""
    if math.isnan(v) or math.isinf(v) or not (-(2.0 ** 63) <= v < 2.0 ** 63):
        return 0
    return round(v)


def int_to_i64(x: int) -> int:
    """any integer (UBIGINT, HUGEINT, UHUGEINT values) -> BIGINT: out of int64 fails (0)"""
    return x if fits_i64(x) else 0


def i32_trunc(x: int) -> int:
    """the int64 result read as int32: low 32 bits, signed"""
    return (x + 2**31) % 2**32 - 2**31


def i32_sat(x: int) -> int:
    return max(I32_MIN, min(I32_MAX, x))


def bool_byte(v) -> int:
    """x != 0: -0.0 gives 0, NaN gives 1"""
    return int(v != 0)


def dec_round(x: int, scale: int) -> int:
    """the stored integer x of a DECIMAL with this scale, rounded half away from zero to an integer"""
    p = 10 ** scale
    q = (abs(x) + p // 2) // p
    return -q if x < 0 else q


def dec_to_i64(x: int, scale: int) -> int:
    """DECIMAL (stored integer x, scale) -> BIGINT: round half away from zero; out of int64 fails (0)"""
    q = dec_round(x, scale)
    return q if fits_i64(q) else 0


# ---------------------------------------------------------------- casts to DOUBLE
def huge_to_f64(x: int) -> float:
    """DuckDB's HUGEINT -> DOUBLE: lower + upper * 2^64 in doubles, upper == -1 negated so small negatives stay exact"""
    lo, hi = x & U64_MAX, x >> 64
    if hi == -1:
        return -float(U64_MAX - lo) - 1.0
    return float(lo) + float(hi) * TWO64


def uhuge_to_f64(x: int) -> float:
    return float(x & U64_MAX) + float(x >> 64) * TWO64


def _trunc_divmod(x: int, p: int):
    """C's truncating division"""
    q = abs(x) // p
    q = -q if x < 0 else q
    return q, x - q * p


def dec_to_f64(x: int, scale: int, width: int) -> float:
    """DuckDB's DECIMAL -> DOUBLE: x / 10^s when x is exact in a double (|x| <= 2^53) or s == 0, else the integer and
    fraction parts converted apart.  Storage up to 18 digits converts int64 -> double; wider storage is a hugeint."""
    conv = float if width <= 18 else huge_to_f64
    p = float(10 ** scale)
    if scale == 0 or abs(x) <= 2**53:
        return conv(x) / p
    q, r = _trunc_divmod(x, 10 ** scale)
    return conv(q) + conv(r) / p


def ulps_apart(a: float, b: float) -> int:
    """distance in units in the last place (finite doubles of the same sign or zero)"""
    ia = int(np.float64(a).view(np.int64))
    ib = int(np.float64(b).view(np.int64))
    ia = ia if ia >= 0 else -(ia & I64_MAX)
    ib = ib if ib >= 0 else -(ib & I64_MAX)
    return abs(ia - ib)


def exact_f64(x: int, scale: int) -> float:
    """the correctly rounded double of x / 10^scale"""
    return float(Fraction(x, 10 ** scale))


# ---------------------------------------------------------------- timestamps, intervals
def ts_us_from_ns(v: int) -> int:
    return v // 1000  # floor: -1 ns is in the microsecond before the epoch


def ts_us_from_ms(v: int) -> int:
    return v * 1000


def ts_us_from_s(v: int) -> int:
    return v * 1_000_000


def month_day_nano(micros: int) -> int:
    return micros * 1000


def _is_leap(y: int) -> bool:
    return (y % 4 == 0 and y % 100 != 0) or y % 400 == 0


@functools.lru_cache(maxsize=None)
def _leaps_from_1970(year: int) -> int:
    """the reference's leap loop: `for ly in 1970..<year`, empty for year <= 1970"""
    return sum(1 for ly in range(1970, year) if _is_leap(ly))


def date_to_days_ref(year: int, month: int, day: int) -> int:
    """the reference's date_to_days (src/duckdb_parsing.mbt:318-338): before 1970 it misses every leap day in
    [year, 1970) (SURVEY.md B.4)"""
    mdays = [31, 29 if _is_leap(year) else 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31]
    return (year - 1970) * 365 + _leaps_from_1970(year) + sum(mdays[: month - 1]) + day - 1


def date_ref(days: int) -> int:
    """typed DATE of the reference: text -> parse_date -> date_to_days for years 1..9999, other days unchanged"""
    y, m, d = civil(days)
    if 1 <= y <= 9999:
        return date_to_days_ref(y, m, d)
    return days


# ---------------------------------------------------------------- renderings
_EPOCH_ORDINAL = datetime.date(1970, 1, 1).toordinal()
_CYCLE_DAYS = 146097  # 400 Gregorian years


def civil(days: int):
    """(year, month, day) of a day number, proleptic Gregorian: shift by whole 400-year cycles into the range of
    datetime.date, convert, shift back"""
    ordinal = days + _EPOCH_ORDINAL
    cycles = (ordinal - 1) // _CYCLE_DAYS
    d = datetime.date.fromordinal(ordinal - cycles * _CYCLE_DAYS)
    return d.year + 400 * cycles, d.month, d.day


def _date_text(days: int) -> str:
    y, m, d = civil(days)
    if y >= 1:
        return f"{y:04d}-{m:02d}-{d:02d}"
    return f"{1 - y:04d}-{m:02d}-{d:02d} (BC)"


def render_int(x: int) -> str:
    return str(x)


def render_decimal(x: int, scale: int) -> str:
    sign = "-" if x < 0 else ""
    p = 10 ** scale
    if scale == 0:
        return sign + str(abs(x))
    return f"{sign}{abs(x) // p}.{abs(x) % p:0{scale}d}"


def render_date(days: int) -> str:
    if days == I32_MAX:
        return "infinity"
    if days == -I32_MAX:
        return "-infinity"
    return _date_text(days)


def _fraction(frac: int, digits: int) -> str:
    s = f"{frac:0{digits}d}".rstrip("0")
    return "." + s if s else ""


def _hms(sod: int) -> str:
    return f"{sod // 3600:02d}:{sod // 60 % 60:02d}:{sod % 60:02d}"


TS_UNITS = {"s": (1, 0), "ms": (1000, 3), "us": (1_000_000, 6), "ns": (1_000_000_000, 9)}


def render_timestamp(v: int, unit: str = "us", tz: bool = False) -> str:
    """TIMESTAMP (unit "us"), TIMESTAMP_TZ (tz), TIMESTAMP_S / _MS / _NS; +-INT64_MAX of the microsecond types are
    DuckDB's infinities"""
    per_sec, digits = TS_UNITS[unit]
    if unit == "us" and v in (I64_MAX, -I64_MAX):
        return "infinity" if v > 0 else "-infinity"
    secs, frac = divmod(v, per_sec)
    days, sod = divmod(secs, 86400)
    return _date_text(days) + " " + _hms(sod) + (_fraction(frac, digits) if frac else "") + ("+00" if tz else "")


def render_time(v: int, unit: str = "us") -> str:
    """TIME / TIME_NS: time of day, 24:00:00 included"""
    per_sec, digits = TS_UNITS[unit]
    secs, frac = divmod(v, per_sec)
    return _hms(secs) + (_fraction(frac, digits) if frac else "")


def render_uuid(x: int) -> str:
    """UUID stored as a hugeint with the top bit flipped"""
    return str(uuid.UUID(int=(x & (2**128 - 1)) ^ 2**127))


def _layout(sign: str, digits: str, exp10: int) -> str:
    """the project's layout of shortest digits (value = 0.digits... as d.ddd * 10^x): fixed notation for
    1e-5 <= |v| < 1e16, always with a fraction ("1.0"); otherwise d.ddde+XX with at least two exponent digits"""
    x = exp10 + len(digits) - 1  # scientific exponent
    if -5 <= x < 16:
        if x >= 0:
            whole = digits[: x + 1].ljust(x + 1, "0")
            frac = digits[x + 1:] or "0"
            return f"{sign}{whole}.{frac}"
        return f"{sign}0.{'0' * (-x - 1)}{digits}"
    mant = digits[0] + ("." + digits[1:] if len(digits) > 1 else "")
    return f"{sign}{mant}e{'-' if x < 0 else '+'}{abs(x):02d}"


def _shortest(text: str, negative: bool) -> str:
    t = Decimal(text).as_tuple()
    digits = "".join(map(str, t.digits)).lstrip("0")
    exp = t.exponent
    if not digits:
        return ("-" if negative else "") + "0.0"
    stripped = digits.rstrip("0")
    exp += len(digits) - len(stripped)
    return _layout("-" if negative else "", stripped, exp)


def _nonfinite(v: float):
    if math.isnan(v):
        return "nan"
    if math.isinf(v):
        return "inf" if v > 0 else "-inf"
    return None


def render_double(v: float) -> str:
    """DOUBLE: the digits of repr(v), Python's shortest round trip"""
    return _nonfinite(v) or _shortest(repr(abs(v)), math.copysign(1.0, v) < 0)


def render_float(v: float) -> str:
    """FLOAT: the float's own shortest digits (numpy's float32 repr), not those of the widened double"""
    f = np.float32(v)
    return _nonfinite(float(f)) or _shortest(str(abs(f)), bool(np.signbit(f)))
