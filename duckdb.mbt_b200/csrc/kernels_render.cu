// K7 render_text: fixed-width DuckDB cells -> their VARCHAR rendering, as duckdb_string_t.
//
// The reference hands every non-VARCHAR cell to libduckdb for text rendering:
// duckdb_value_varchar in the result path (src/duckdb_native.c:224-238, and :2478 / :2715 for the
// "string" getters that its schema JSON prescribes for DATE / DECIMAL / TIMESTAMP / ... columns,
// :2314-2339) and duckdb_value_to_string in the chunk path (:305-318, :611-661).  Here one thread
// renders one cell into a 48-byte slot (80 for INTERVAL) and emits a 16-byte string_t (<= 12 bytes inlined, else
// prefix + pointer to the slot), so the rendered column then flows through the same
// string_batch_kernel (utf8 offsets + data, or the reference's NUL-terminated blob) as a VARCHAR
// column.  Formats follow DuckDB 1.4's renderings pinned by src/duckdb_fixture_cases.mbt
// (ints :27-32,83-102, HUGEINT sums :34-37,174-177, DATE :41-46, TIME :48-51, TIMESTAMP :55-67, DECIMAL :69-81).

#include "dmb_common.cuh"

namespace dmb {

template <int SLOT>
struct TextBuf {
  char s[SLOT];
  int n;
  __device__ __forceinline__ void push(char c) { if (n < SLOT) s[n++] = c; }
  __device__ __forceinline__ void push_str(const char *p) { while (*p) push(*p++); }
  // unsigned decimal, at least `min_digits` digits (zero padded)
  __device__ __forceinline__ void push_u64(uint64_t v, int min_digits) {
    char tmp[20];
    int k = 0;
    do { tmp[k++] = (char)('0' + (int)(v % 10ull)); v /= 10ull; } while (v != 0ull);
    for (int i = k; i < min_digits; ++i) push('0');
    while (k > 0) push(tmp[--k]);
  }
};

__device__ __forceinline__ int64_t floor_div64(int64_t a, int64_t b) {
  int64_t q = a / b;
  return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}

template <class TB>
__device__ __forceinline__ void render_i64(TB &t, int64_t v) {
  if (v < 0) { t.push('-'); t.push_u64((uint64_t)0 - (uint64_t)v, 1); } else t.push_u64((uint64_t)v, 1);
}

// DECIMAL(w, scale) stored as an integer: sign, integer part, '.', exactly `scale` fraction digits
template <class TB>
__device__ __forceinline__ void render_decimal(TB &t, int64_t v, int scale) {
  const bool neg = v < 0;
  uint64_t a = neg ? (uint64_t)0 - (uint64_t)v : (uint64_t)v;
  if (neg) t.push('-');
  if (scale <= 0) { t.push_u64(a, 1); return; }
  uint64_t p = 1;
  for (int i = 0; i < scale; ++i) p *= 10ull;
  t.push_u64(a / p, 1);
  t.push('.');
  t.push_u64(a % p, scale);
}

// proleptic Gregorian date: YYYY-MM-DD, more digits past year 9999, "(BC)" suffix before year 1
template <class TB>
__device__ __forceinline__ void render_date(TB &t, int64_t days) {
  int64_t z = days + 719468;
  const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  const int64_t doe = z - era * 146097;
  const int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  const int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  const int64_t mp = (5 * doy + 2) / 153;
  const int d = (int)(doy - (153 * mp + 2) / 5 + 1);
  const int m = (int)(mp < 10 ? mp + 3 : mp - 9);
  const int64_t y = yoe + era * 400 + (m <= 2 ? 1 : 0);
  const bool bc = y < 1;
  t.push_u64((uint64_t)(bc ? 1 - y : y), 4);
  t.push('-');
  t.push_u64((uint64_t)m, 2);
  t.push('-');
  t.push_u64((uint64_t)d, 2);
  if (bc) t.push_str(" (BC)");
}

// v in units of 1/unit_per_sec seconds since the epoch; fraction digits trimmed of trailing zeros
template <class TB>
__device__ __forceinline__ void render_timestamp(TB &t, int64_t v, int64_t unit_per_sec, bool tz) {
  const int64_t secs = floor_div64(v, unit_per_sec);
  const int64_t frac = v - secs * unit_per_sec;
  const int64_t days = floor_div64(secs, 86400);
  const int64_t sod = secs - days * 86400;
  render_date(t, (int64_t)(int32_t)days);  // the oracle narrows the day number to int32 like DuckDB's date_t
  t.push(' ');
  t.push_u64((uint64_t)(sod / 3600), 2);
  t.push(':');
  t.push_u64((uint64_t)(sod / 60 % 60), 2);
  t.push(':');
  t.push_u64((uint64_t)(sod % 60), 2);
  if (frac != 0) {
    int digits = unit_per_sec == 1000 ? 3 : (unit_per_sec == 1000000 ? 6 : 9);
    uint64_t f = (uint64_t)frac;
    while (digits > 0 && f % 10ull == 0ull) { f /= 10ull; --digits; }
    t.push('.');
    t.push_u64(f, digits);
  }
  if (tz) t.push_str("+00");
}

// TIME: HH:MM:SS[.fraction], fraction digits trimmed of trailing zeros (fixture src/duckdb_fixture_cases.mbt:48-51)
template <class TB>
__device__ __forceinline__ void render_time(TB &t, int64_t v, int64_t unit_per_sec) {
  const int64_t secs = v / unit_per_sec, frac = v % unit_per_sec;
  t.push_u64((uint64_t)(secs / 3600), 2);
  t.push(':');
  t.push_u64((uint64_t)(secs / 60 % 60), 2);
  t.push(':');
  t.push_u64((uint64_t)(secs % 60), 2);
  if (frac != 0) {
    int digits = unit_per_sec == 1000000 ? 6 : 9;
    uint64_t f = (uint64_t)frac;
    while (digits > 0 && f % 10ull == 0ull) { f /= 10ull; --digits; }
    t.push('.');
    t.push_u64(f, digits);
  }
}

// 128-bit integers (HUGEINT: what SUM() of an integer column returns, fixtures :34-37; UHUGEINT;
// DECIMAL(19..38, scale)): three base-10^19 limbs, '.' before the last `scale` digits
template <class TB>
__device__ __forceinline__ void render_i128(TB &t, unsigned __int128 u, bool is_signed, int scale) {
  const bool neg = is_signed && (__int128)u < 0;
  unsigned __int128 a = neg ? (unsigned __int128)0 - u : u;
  const unsigned __int128 kP19 = 10000000000000000000ull;
  char d[40];  // least significant digit first
  int n = 0;
#pragma unroll 1
  for (int limb = 0; limb < 3; ++limb) {
    uint64_t r = (uint64_t)(a % kP19);
    a /= kP19;
    const bool last = a == 0;
    for (int i = 0; i < 19 && n < 39; ++i) {
      if (last && r == 0ull && i > 0) break;
      d[n++] = (char)('0' + (int)(r % 10ull));
      r /= 10ull;
    }
    if (last) break;
  }
  if (n == 0) d[n++] = '0';
  while (n <= scale && n < 40) d[n++] = '0';  // at least one digit before the point
  if (neg) t.push('-');
  for (int i = n - 1; i >= 0; --i) {
    t.push(d[i]);
    if (scale > 0 && i == scale) t.push('.');
  }
}

// ---- DOUBLE / FLOAT: shortest decimal that reads back as the same double / float (what DuckDB's fmt-based
// cast prints: "3.5", "5.333333333333333", src/duckdb_fixture_cases.mbt:20-25,167-172,216-221),
// by Ryu (Ulf Adams, PLDI 2018): one 64x128-bit multiplication by a tabulated power of 5 gives the
// decimal images of the value and of its two rounding-interval ends, then digits are dropped
// while the ends still differ.  Tables: ryu_tables.inc (gen/make_ryu_tables.py).
#include "ryu_tables.inc"

__device__ __forceinline__ uint64_t ryu_mul_shift(uint64_t m, const unsigned long long *mul, int j) {
  const unsigned __int128 b0 = (unsigned __int128)m * __ldg(mul);
  const unsigned __int128 b2 = (unsigned __int128)m * __ldg(mul + 1);
  return (uint64_t)(((b0 >> 64) + b2) >> (j - 64));
}
__device__ __forceinline__ bool ryu_multiple_of_pow5(uint64_t v, int p) {
  int c = 0;
  while (v != 0ull && v % 5ull == 0ull) { v /= 5ull; ++c; }
  return c >= p;
}
// bits of a finite non-zero double -> (digits, exponent): value = digits * 10^exponent, digits shortest
__device__ __forceinline__ uint64_t ryu_shortest(uint64_t bits, int &exp10) {
  const uint64_t ieee_m = bits & ((1ull << 52) - 1ull);
  const int ieee_e = (int)((bits >> 52) & 0x7ffu);
  int e2;
  uint64_t m2;
  if (ieee_e == 0) { e2 = 1 - 1023 - 52 - 2; m2 = ieee_m; }
  else { e2 = ieee_e - 1023 - 52 - 2; m2 = (1ull << 52) | ieee_m; }
  const bool accept = (m2 & 1ull) == 0ull;  // round-to-even: the interval ends themselves read back
  const uint64_t mv = 4ull * m2;
  const uint32_t mm_shift = (ieee_m != 0ull || ieee_e <= 1) ? 1u : 0u;  // below a power of two the interval is half as wide
  uint64_t vr, vp, vm;
  int e10;
  bool vm_tz = false, vr_tz = false;
  if (e2 >= 0) {
    const int q = ((e2 * 78913) >> 18) - (e2 > 3 ? 1 : 0);
    e10 = q;
    const int k = 125 + (((q * 1217359) >> 19) + 1) - 1;
    const int i = -e2 + q + k;
    const unsigned long long *mul = kRyuPow5InvSplit[q];
    vr = ryu_mul_shift(mv, mul, i);
    vp = ryu_mul_shift(mv + 2ull, mul, i);
    vm = ryu_mul_shift(mv - 1ull - mm_shift, mul, i);
    if (q <= 21) {
      if (mv % 5ull == 0ull) vr_tz = ryu_multiple_of_pow5(mv, q);
      else if (accept) vm_tz = ryu_multiple_of_pow5(mv - 1ull - mm_shift, q);
      else vp -= ryu_multiple_of_pow5(mv + 2ull, q) ? 1ull : 0ull;
    }
  } else {
    const int q = (((-e2) * 732923) >> 20) - (-e2 > 1 ? 1 : 0);
    e10 = q + e2;
    const int i = -e2 - q;
    const int k = (((i * 1217359) >> 19) + 1) - 125;
    const int j = q - k;
    const unsigned long long *mul = kRyuPow5Split[i];
    vr = ryu_mul_shift(mv, mul, j);
    vp = ryu_mul_shift(mv + 2ull, mul, j);
    vm = ryu_mul_shift(mv - 1ull - mm_shift, mul, j);
    if (q <= 1) {
      vr_tz = true;
      if (accept) vm_tz = mm_shift == 1u;
      else --vp;
    } else if (q < 63) {
      vr_tz = (mv & ((1ull << q) - 1ull)) == 0ull;
    }
  }
  int removed = 0;
  uint32_t last = 0;
  uint64_t out;
  if (vm_tz || vr_tz) {  // rare: exact decimal images, ties must be seen
    while (vp / 10ull > vm / 10ull) {
      vm_tz = vm_tz && vm % 10ull == 0ull;
      vr_tz = vr_tz && last == 0u;
      last = (uint32_t)(vr % 10ull);
      vr /= 10ull; vp /= 10ull; vm /= 10ull;
      ++removed;
    }
    if (vm_tz) {
      while (vm % 10ull == 0ull) {
        vr_tz = vr_tz && last == 0u;
        last = (uint32_t)(vr % 10ull);
        vr /= 10ull; vp /= 10ull; vm /= 10ull;
        ++removed;
      }
    }
    if (vr_tz && last == 5u && vr % 2ull == 0ull) last = 4u;  // exactly half: round to even
    out = vr + (((vr == vm && (!accept || !vm_tz)) || last >= 5u) ? 1ull : 0ull);
  } else {
    bool round_up = false;
    while (vp / 10ull > vm / 10ull) {
      round_up = vr % 10ull >= 5ull;
      vr /= 10ull; vp /= 10ull; vm /= 10ull;
      ++removed;
    }
    out = vr + ((vr == vm || round_up) ? 1ull : 0ull);
  }
  exp10 = e10 + removed;
  return out;
}

// FLOAT: Ryu's float form (f2s), the same steps on a 24-bit significand with 32-bit decimal images.  Its
// multipliers are the high words of the double tables (61 significant bits; the inverse ones + 1).
__device__ __forceinline__ uint32_t ryu_mul_shift32(uint32_t m, uint64_t factor, int shift) {
  const uint64_t sum = (((uint64_t)m * (uint32_t)factor) >> 32) + (uint64_t)m * (uint32_t)(factor >> 32);
  return (uint32_t)(sum >> (shift - 32));
}
__device__ __forceinline__ uint32_t ryu_pow5_inv32(uint32_t m, int q, int j) { return ryu_mul_shift32(m, __ldg(&kRyuPow5InvSplit[q][1]) + 1ull, j); }
__device__ __forceinline__ uint32_t ryu_pow5_32(uint32_t m, int i, int j) { return ryu_mul_shift32(m, __ldg(&kRyuPow5Split[i][1]), j); }
__device__ __forceinline__ int ryu_pow5_bits(int e) { return ((e * 1217359) >> 19) + 1; }
// bits of a finite non-zero float -> (digits, exponent): value = digits * 10^exponent, digits shortest
__device__ __forceinline__ uint32_t ryu_shortest_f32(uint32_t bits, int &exp10) {
  constexpr int kBits = 61;  // 125 - 64
  const uint32_t ieee_m = bits & ((1u << 23) - 1u);
  const int ieee_e = (int)((bits >> 23) & 0xffu);
  int e2;
  uint32_t m2;
  if (ieee_e == 0) { e2 = 1 - 127 - 23 - 2; m2 = ieee_m; }
  else { e2 = ieee_e - 127 - 23 - 2; m2 = (1u << 23) | ieee_m; }
  const bool accept = (m2 & 1u) == 0u;
  const uint32_t mv = 4u * m2, mp = mv + 2u;
  const uint32_t mm = mv - 1u - ((ieee_m != 0u || ieee_e <= 1) ? 1u : 0u);
  uint32_t vr, vp, vm, last = 0;
  int e10;
  bool vm_tz = false, vr_tz = false;
  auto pow5_multiple = [](uint32_t v, int p) { int c = 0; while (v != 0u && v % 5u == 0u) { v /= 5u; ++c; } return c >= p; };
  if (e2 >= 0) {
    const int q = (e2 * 78913) >> 18;
    e10 = q;
    const int i = -e2 + q + kBits + ryu_pow5_bits(q) - 1;
    vr = ryu_pow5_inv32(mv, q, i);
    vp = ryu_pow5_inv32(mp, q, i);
    vm = ryu_pow5_inv32(mm, q, i);
    if (q != 0 && (vp - 1u) / 10u <= vm / 10u)  // the loop below may not run: one removed digit is still needed
      last = ryu_pow5_inv32(mv, q - 1, -e2 + q - 1 + kBits + ryu_pow5_bits(q - 1) - 1) % 10u;
    if (q <= 9) {
      if (mv % 5u == 0u) vr_tz = pow5_multiple(mv, q);
      else if (accept) vm_tz = pow5_multiple(mm, q);
      else vp -= pow5_multiple(mp, q) ? 1u : 0u;
    }
  } else {
    const int q = ((-e2) * 732923) >> 20;
    e10 = q + e2;
    const int i = -e2 - q;
    const int j = q - (ryu_pow5_bits(i) - kBits);
    vr = ryu_pow5_32(mv, i, j);
    vp = ryu_pow5_32(mp, i, j);
    vm = ryu_pow5_32(mm, i, j);
    if (q != 0 && (vp - 1u) / 10u <= vm / 10u)
      last = ryu_pow5_32(mv, i + 1, q - 1 - (ryu_pow5_bits(i + 1) - kBits)) % 10u;
    if (q <= 1) {
      vr_tz = true;
      if (accept) vm_tz = mm == mv - 2u;
      else --vp;
    } else if (q < 31) {
      vr_tz = (mv & ((1u << (q - 1)) - 1u)) == 0u;
    }
  }
  int removed = 0;
  uint32_t out;
  if (vm_tz || vr_tz) {
    while (vp / 10u > vm / 10u) {
      vm_tz = vm_tz && vm % 10u == 0u;
      vr_tz = vr_tz && last == 0u;
      last = vr % 10u;
      vr /= 10u; vp /= 10u; vm /= 10u;
      ++removed;
    }
    if (vm_tz) {
      while (vm % 10u == 0u) {
        vr_tz = vr_tz && last == 0u;
        last = vr % 10u;
        vr /= 10u; vp /= 10u; vm /= 10u;
        ++removed;
      }
    }
    if (vr_tz && last == 5u && vr % 2u == 0u) last = 4u;  // exactly half: round to even
    out = vr + (((vr == vm && (!accept || !vm_tz)) || last >= 5u) ? 1u : 0u);
  } else {
    while (vp / 10u > vm / 10u) {
      last = vr % 10u;
      vr /= 10u; vp /= 10u; vm /= 10u;
      ++removed;
    }
    out = vr + ((vr == vm || last >= 5u) ? 1u : 0u);
  }
  exp10 = e10 + removed;
  return out;
}

// fmt-style layout of the digits: fixed notation for 1e-5 <= |v| < 1e16 (always with a fraction:
// "1.0"), else d.ddde+XX (at least two exponent digits).  DOUBLE takes the double's shortest digits,
// FLOAT the float's own ("0.1", not the widened double's "0.10000000149011612"), as DuckDB prints them.
template <class TB>
__device__ __forceinline__ void render_double(TB &t, double v, bool is_float) {
  const uint64_t bits = (uint64_t)__double_as_longlong(v);
  if (((bits >> 52) & 0x7ffu) == 0x7ffu) {
    if (bits & ((1ull << 52) - 1ull)) t.push_str("nan");
    else t.push_str((bits >> 63) ? "-inf" : "inf");
    return;
  }
  uint64_t digits = 0;
  int e = 0;
  if (bits & ~(1ull << 63)) digits = is_float ? ryu_shortest_f32(__float_as_uint((float)v), e) : ryu_shortest(bits, e);
  while (digits != 0ull && digits % 10ull == 0ull) { digits /= 10ull; ++e; }
  char m[20];  // most significant digit first
  int nd = 0;
  {
    char r[20];
    uint64_t x = digits;
    do { r[nd++] = (char)('0' + (int)(x % 10ull)); x /= 10ull; } while (x != 0ull);
    for (int i = 0; i < nd; ++i) m[i] = r[nd - 1 - i];
  }
  const int x10 = e + nd - 1;  // scientific exponent
  if (bits >> 63) t.push('-');
  if (x10 >= -5 && x10 < 16) {
    if (x10 >= 0) {
      for (int i = 0; i <= x10; ++i) t.push(i < nd ? m[i] : '0');
      t.push('.');
      if (nd > x10 + 1) { for (int i = x10 + 1; i < nd; ++i) t.push(m[i]); }
      else t.push('0');
    } else {
      t.push('0');
      t.push('.');
      for (int i = 0; i < -x10 - 1; ++i) t.push('0');
      for (int i = 0; i < nd; ++i) t.push(m[i]);
    }
    return;
  }
  t.push(m[0]);
  if (nd > 1) { t.push('.'); for (int i = 1; i < nd; ++i) t.push(m[i]); }
  t.push('e');
  t.push(x10 < 0 ? '-' : '+');
  t.push_u64((uint64_t)(x10 < 0 ? -x10 : x10), 2);
}

// UUID: DuckDB keeps a UUID as a hugeint whose top bit is flipped (so that UUIDs order like signed hugeints);
// text is lowercase hex 8-4-4-4-12.  UNPINNED (no reference fixture holds a UUID).
template <class TB>
__device__ __forceinline__ void render_uuid(TB &t, unsigned __int128 u) {
  const uint64_t hi = (uint64_t)(u >> 64) ^ (1ull << 63), lo = (uint64_t)u;
  auto hex = [&](uint64_t v, int digits) {
    for (int i = digits - 1; i >= 0; --i) t.push("0123456789abcdef"[(v >> (4 * i)) & 15ull]);
  };
  hex(hi >> 32, 8); t.push('-');
  hex(hi >> 16, 4); t.push('-');
  hex(hi, 4); t.push('-');
  hex(lo >> 48, 4); t.push('-');
  hex(lo, 12);
}

// TIME WITH TIME ZONE: bits = micros << 24 | (57599 - offset seconds); text = TIME, then +HH / -HH, ":MM" and ":SS"
// only when non-zero.  UNPINNED.
template <class TB>
__device__ __forceinline__ void render_time_tz(TB &t, uint64_t bits) {
  render_time(t, (int64_t)(bits >> 24), 1000000);
  int off = 57599 - (int)(bits & 0xffffffull);
  t.push(off < 0 ? '-' : '+');
  if (off < 0) off = -off;
  t.push_u64((uint64_t)(off / 3600), 2);
  const int mm = off % 3600 / 60, ss = off % 60;
  if (mm) { t.push(':'); t.push_u64((uint64_t)mm, 2); }
  if (ss) { t.push(':'); t.push_u64((uint64_t)ss, 2); }
}

// INTERVAL {months, days, micros}: "Y year[s] M month[s] D day[s] [-]HH:MM:SS[.ffffff]", zero parts left out,
// "00:00:00" when everything is zero; unit names take an 's' unless the count is +-1.  UNPINNED.
template <class TB>
__device__ __forceinline__ void render_interval(TB &t, int32_t months, int32_t days, int64_t micros) {
  auto part = [&](int64_t v, const char *name) {
    if (v == 0) return;
    if (t.n) t.push(' ');
    render_i64(t, v);
    t.push_str(name);
    if (v != 1 && v != -1) t.push('s');
  };
  const int32_t years = months / 12;
  part(years, " year");
  part(months - years * 12, " month");
  part(days, " day");
  if (micros != 0) {
    if (t.n) t.push(' ');
    int64_t m = micros;  // kept non-positive: INT64_MIN has no positive twin
    if (m < 0) t.push('-'); else m = -m;
    const int64_t hour = -(m / 3600000000ll);
    m += hour * 3600000000ll;
    const int64_t min = -(m / 60000000ll);
    m += min * 60000000ll;
    const int64_t sec = -(m / 1000000ll);
    m += sec * 1000000ll;
    t.push_u64((uint64_t)hour, 2);
    t.push(':');
    t.push_u64((uint64_t)min, 2);
    t.push(':');
    t.push_u64((uint64_t)sec, 2);
    uint64_t f = (uint64_t)(-m);
    if (f) {
      int digits = 6;
      while (f % 10ull == 0ull) { f /= 10ull; --digits; }
      t.push('.');
      t.push_u64(f, digits);
    }
  } else if (t.n == 0) {
    t.push_str("00:00:00");
  }
}

template <int SLOT>
__global__ void __launch_bounds__(kThreads)
render_text_kernel(dmb_render_job job, const uint32_t *__restrict__ counts, int64_t nchunks) {
  for (int64_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const int count = (int)__ldg(counts + c);
    const dmb_vec_desc vd = job.vecs[c];
    const uint8_t *in = reinterpret_cast<const uint8_t *>(job.in_data) + vd.data_off;
    const uint64_t *mask = vd.val_off < 0 ? nullptr : job.in_validity + vd.val_off;
    for (int i = threadIdx.x; i < count; i += kThreads) {
      const int64_t slot = c * (int64_t)kVec + i;
      uint4 e = make_uint4(0, 0, 0, 0);
      const bool valid = mask ? ((__ldg(mask + (i >> 6)) >> (i & 63)) & 1ull) : true;
      if (valid) {
        TextBuf<SLOT> t;
        t.n = 0;
        int64_t v = 0;
        uint64_t u = 0;
        switch (job.phys) {
          case DMB_PHYS_BOOL: case DMB_PHYS_U8: u = in[i]; v = (int64_t)u; break;
          case DMB_PHYS_I8: v = reinterpret_cast<const int8_t *>(in)[i]; break;
          case DMB_PHYS_I16: v = reinterpret_cast<const int16_t *>(in)[i]; break;
          case DMB_PHYS_U16: u = reinterpret_cast<const uint16_t *>(in)[i]; v = (int64_t)u; break;
          case DMB_PHYS_I32: v = reinterpret_cast<const int32_t *>(in)[i]; break;
          case DMB_PHYS_U32: u = reinterpret_cast<const uint32_t *>(in)[i]; v = (int64_t)u; break;
          case DMB_PHYS_I64: v = reinterpret_cast<const int64_t *>(in)[i]; break;
          case DMB_PHYS_U64: u = reinterpret_cast<const uint64_t *>(in)[i]; v = (int64_t)u; break;
          default: break;
        }
        double fv = 0.0;
        if (job.phys == DMB_PHYS_F64) fv = reinterpret_cast<const double *>(in)[i];
        if (job.phys == DMB_PHYS_F32) fv = (double)reinterpret_cast<const float *>(in)[i];  // exact; rendered with the float's digits
        unsigned __int128 wide = 0;
        if (job.phys == DMB_PHYS_I128 || job.phys == DMB_PHYS_U128 || job.phys == DMB_PHYS_INTERVAL) {
          const uint4 q = reinterpret_cast<const uint4 *>(in)[i];
          wide = ((unsigned __int128)(((uint64_t)q.w << 32) | q.z) << 64) | (((uint64_t)q.y << 32) | q.x);
        }
        switch (job.type_id) {
          case DMB_TYPE_BOOLEAN: t.push_str(u ? "true" : "false"); break;
          case DMB_TYPE_UBIGINT: t.push_u64(u, 1); break;
          // DuckDB's infinite DATE is +-INT32_MAX and its infinite TIMESTAMP / TIMESTAMPTZ +-INT64_MAX; they print as words
          case DMB_TYPE_DATE:
            if (v == 2147483647ll || v == -2147483647ll) t.push_str(v < 0 ? "-infinity" : "infinity"); else render_date(t, v);
            break;
          case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_TZ:
            if (v == INT64_MAX || v == -INT64_MAX) t.push_str(v < 0 ? "-infinity" : "infinity");
            else render_timestamp(t, v, 1000000, job.type_id == DMB_TYPE_TIMESTAMP_TZ);
            break;
          case DMB_TYPE_TIMESTAMP_S: render_timestamp(t, v, 1, false); break;
          case DMB_TYPE_TIMESTAMP_MS: render_timestamp(t, v, 1000, false); break;
          case DMB_TYPE_TIMESTAMP_NS: render_timestamp(t, v, 1000000000, false); break;
          case DMB_TYPE_DECIMAL:
            if (job.phys == DMB_PHYS_I128) render_i128(t, wide, true, job.dec_scale); else render_decimal(t, v, job.dec_scale);
            break;
          case DMB_TYPE_FLOAT: case DMB_TYPE_DOUBLE: render_double(t, fv, job.type_id == DMB_TYPE_FLOAT); break;
          case DMB_TYPE_HUGEINT: render_i128(t, wide, true, 0); break;
          case DMB_TYPE_UHUGEINT: render_i128(t, wide, false, 0); break;
          case DMB_TYPE_TIME: render_time(t, v, 1000000); break;
          case DMB_TYPE_TIME_NS: render_time(t, v, 1000000000); break;
          case DMB_TYPE_TIME_TZ: render_time_tz(t, u); break;
          case DMB_TYPE_UUID: render_uuid(t, wide); break;
          case DMB_TYPE_INTERVAL: render_interval(t, (int32_t)(uint32_t)wide, (int32_t)(uint32_t)(wide >> 32), (int64_t)(uint64_t)(wide >> 64)); break;
          default: render_i64(t, v); break;  // TINYINT .. BIGINT, UTINYINT .. UINTEGER
        }
        // string_t: length, then 12 inlined bytes or 4-byte prefix + pointer to the slot
        uint32_t w[SLOT / 4];
#pragma unroll
        for (int k = 0; k < SLOT / 4; ++k) {
          uint32_t x = 0;
#pragma unroll
          for (int bb = 0; bb < 4; ++bb) x |= (4 * k + bb < t.n ? (uint32_t)(uint8_t)t.s[4 * k + bb] : 0u) << (8 * bb);
          w[k] = x;
        }
        e.x = (uint32_t)t.n;
        e.y = w[0];
        if (t.n <= 12) {
          e.z = w[1];
          e.w = w[2];
        } else {
          const uint64_t p = job.heap_host_base + (uint64_t)slot * SLOT;
          e.z = (uint32_t)p;
          e.w = (uint32_t)(p >> 32);
          uint4 *dst = reinterpret_cast<uint4 *>(job.out_heap + (uint64_t)slot * SLOT);
#pragma unroll
          for (int k = 0; k < SLOT / 16; ++k) dst[k] = make_uint4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
        }
      }
      reinterpret_cast<uint4 *>(job.out)[slot] = e;
    }
  }
}

}  // namespace dmb

using namespace dmb;

// bytes of out_heap per row: the longest rendering of the type, rounded up to 16 (INTERVAL: up to 70 characters)
extern "C" int32_t dmb_render_slot_bytes(int32_t type_id) {
  return type_id == DMB_TYPE_INTERVAL ? DMB_RENDER_SLOT_BYTES_WIDE : DMB_RENDER_SLOT_BYTES;
}

namespace dmb {
// BLOB -> its VARCHAR cast (DuckDB Blob::ToString): printable ASCII except backslash and the two quote characters is
// copied, every other byte becomes \xHH (upper-case hex).  One thread per row of a DENSE utf8-style column (offsets +
// data, what dmb_dev_string_batch produced from the BLOB column); row i's escaped bytes go to out_heap + 4 * offsets[i]
// (a byte grows to at most four), the row's string_t refers to them.  Replaces libduckdb's duckdb_value_varchar on a BLOB
// cell (src/duckdb_native.c:224-238, :2478, :2715).  UNPINNED: no reference test reads a BLOB as text.
__global__ void __launch_bounds__(kThreads)
blob_escape_kernel(const int32_t *__restrict__ offsets, const uint8_t *__restrict__ data, int64_t nrows, dmb_string_t *__restrict__ out,
                   uint8_t *__restrict__ out_heap, uint64_t heap_host_base) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < nrows; i += (int64_t)gridDim.x * kThreads) {
    const uint32_t o0 = (uint32_t)offsets[i], o1 = (uint32_t)offsets[i + 1];
    uint8_t *dst = out_heap + 4ull * o0;
    uint32_t n = 0;
    for (uint32_t q = o0; q < o1; ++q) {
      const uint8_t c = data[q];
      if (c >= 32 && c <= 126 && c != '\\' && c != '\'' && c != '"') {
        dst[n++] = c;
      } else {
        const char *hex = "0123456789ABCDEF";
        dst[n++] = '\\';
        dst[n++] = 'x';
        dst[n++] = (uint8_t)hex[c >> 4];
        dst[n++] = (uint8_t)hex[c & 15];
      }
    }
    uint4 e = make_uint4(n, 0, 0, 0);
    uint8_t *eb = reinterpret_cast<uint8_t *>(&e);
    if (n <= 12u) {
      for (uint32_t k = 0; k < n; ++k) eb[4 + k] = dst[k];
    } else {
      for (uint32_t k = 0; k < 4; ++k) eb[4 + k] = dst[k];
      const uint64_t p = heap_host_base + 4ull * o0;
      e.z = (uint32_t)p;
      e.w = (uint32_t)(p >> 32);
    }
    reinterpret_cast<uint4 *>(out)[i] = e;
  }
}

}  // namespace dmb
using namespace dmb;

extern "C" int32_t dmb_dev_blob_escape(const int32_t *offsets, const uint8_t *data, int64_t nrows, dmb_string_t *out, uint8_t *out_heap,
                                       uint64_t heap_host_base, void *stream) {
  if (nrows <= 0) return 0;
  const int64_t blocks = (nrows + kThreads - 1) / kThreads;
  const int grid = (int)(blocks < (int64_t)kNumSMs * 16 ? blocks : (int64_t)kNumSMs * 16);
  blob_escape_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(offsets, data, nrows, out, out_heap, heap_host_base);
  return check_cuda(cudaGetLastError(), "blob_escape_kernel launch");
}

extern "C" int32_t dmb_render_supported(int32_t type_id, int32_t phys) {
  switch (type_id) {
    case DMB_TYPE_BOOLEAN: case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: case DMB_TYPE_BIGINT:
    case DMB_TYPE_UTINYINT: case DMB_TYPE_USMALLINT: case DMB_TYPE_UINTEGER: case DMB_TYPE_UBIGINT: case DMB_TYPE_DATE:
    case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_TZ: case DMB_TYPE_TIMESTAMP_S: case DMB_TYPE_TIMESTAMP_MS:
    case DMB_TYPE_TIMESTAMP_NS:
      return 1;
    case DMB_TYPE_TIME: case DMB_TYPE_TIME_NS:
      return phys == DMB_PHYS_I64;
    case DMB_TYPE_FLOAT: return phys == DMB_PHYS_F32;
    case DMB_TYPE_DOUBLE: return phys == DMB_PHYS_F64;
    case DMB_TYPE_HUGEINT: return phys == DMB_PHYS_I128;
    case DMB_TYPE_UHUGEINT: return phys == DMB_PHYS_U128;
    case DMB_TYPE_DECIMAL: return phys == DMB_PHYS_I16 || phys == DMB_PHYS_I32 || phys == DMB_PHYS_I64 || phys == DMB_PHYS_I128;
    case DMB_TYPE_TIME_TZ: return phys == DMB_PHYS_U64 || phys == DMB_PHYS_I64;
    case DMB_TYPE_UUID: return phys == DMB_PHYS_U128 || phys == DMB_PHYS_I128;
    case DMB_TYPE_INTERVAL: return phys == DMB_PHYS_INTERVAL;
    default: return 0;  // BLOB and nested types: not rendered on the device
  }
}

extern "C" int32_t dmb_dev_render_text(const dmb_render_job *job, const uint32_t *counts, int64_t nchunks, void *stream) {
  if (!job) { set_error("dmb_dev_render_text: job is null"); return -1; }
  if (!dmb_render_supported(job->type_id, job->phys)) { set_error("dmb_dev_render_text: no device renderer for type %d", job->type_id); return -1; }
  if (nchunks <= 0) return 0;
  const int64_t max_grid = (int64_t)kNumSMs * 8;
  const int grid = (int)(nchunks < max_grid ? nchunks : max_grid);
  if (dmb_render_slot_bytes(job->type_id) == DMB_RENDER_SLOT_BYTES_WIDE) render_text_kernel<DMB_RENDER_SLOT_BYTES_WIDE><<<grid, kThreads, 0, (cudaStream_t)stream>>>(*job, counts, nchunks);
  else render_text_kernel<DMB_RENDER_SLOT_BYTES><<<grid, kThreads, 0, (cudaStream_t)stream>>>(*job, counts, nchunks);
  return check_cuda(cudaGetLastError(), "render_text_kernel launch");
}
