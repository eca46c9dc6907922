// K1 validity_to_arrow + K2 fixed_copy + K3 bool_pack + K4 decimal_widen/hugeint/date_ts casts,
// fused: every fixed-width column of a chunk batch is converted by ONE launch
// (SURVEY.md §2.2).  HBM-bound byte movement: 128-bit streaming loads/stores, no tensor cores.
//
// Work item = (column job, chunk index i).  An item does two things:
//   phase A  chunk i's payload  -> contiguous output values at row_off[i]   (chunk-centric)
//   phase B  output tile i (rows [2048 i, 2048 i + 2048)) of the validity bitmap / byte
//            validity / null count                                            (tile-centric)
// Phase B is tile-centric so that bitmap words are written whole even when short chunks put
// chunk boundaries at arbitrary bit offsets (no atomics, no pre-zeroing).
//
// Replaces the reference's per-cell loops src/duckdb_native.c:2379-2387 (int32), :2413-2419
// (int64), :2445-2451 (double), :2537-2543 (bool), their nullable twins :2597-2606, :2635-2644,
// :2673-2682, :2785-2794, and the per-cell validity test :520-535.

#include "dmb_common.cuh"

namespace dmb {

constexpr int kGroupU = 4;  // 16-byte vectors in flight per thread in the narrow-type group path

// ------------------------------------------------------------------ value conversions
// duckdb_value_int64 semantics (libduckdb, un-vendored; cast failure yields 0).  Only the
// same-family integer cases are pinned by reference tests (SURVEY.md §8c); the float and
// 128-bit sources follow DuckDB's documented TryCast (round-to-nearest-even, range check).
template <typename S>
__device__ __forceinline__ int64_t to_i64(S v) { return (int64_t)v; }
template <>
__device__ __forceinline__ int64_t to_i64<uint64_t>(uint64_t v) {
  return v > 0x7fffffffffffffffull ? 0 : (int64_t)v;
}
template <>
__device__ __forceinline__ int64_t to_i64<double>(double v) {
  if (!(v >= -9223372036854775808.0 && v < 9223372036854775808.0)) return 0;
  return __double2ll_rn(v);
}
template <>
__device__ __forceinline__ int64_t to_i64<float>(float v) {
  if (!(v >= -9223372036854775808.0f && v < 9223372036854775808.0f)) return 0;
  return __float2ll_rn(v);
}
template <>
__device__ __forceinline__ int64_t to_i64<i128>(i128 v) {
  bool fits = (v.hi == 0 && (int64_t)v.lo >= 0) || (v.hi == -1 && (int64_t)v.lo < 0);
  return fits ? (int64_t)v.lo : 0;
}

template <>
__device__ __forceinline__ int64_t to_i64<u128>(u128 v) {  // UHUGEINT: fits iff upper == 0 and lower <= INT64_MAX
  return (v.hi == 0 && v.lo <= 0x7fffffffffffffffull) ? (int64_t)v.lo : 0;
}

template <typename S>
__device__ __forceinline__ double to_f64(S v) { return (double)v; }
// DuckDB Hugeint::TryCast<double> (CastBigintToFloating): lower + upper * 2^64 in double arithmetic, with the
// special case for upper == -1 that keeps small negative numbers exact.  UNPINNED (SUM() results read through
// duckdb_value_double, src/duckdb_native.c:2449).
template <>
__device__ __forceinline__ double to_f64<i128>(i128 v) {
  if (v.hi == -1) return -(double)(0xffffffffffffffffull - v.lo) - 1.0;
  return (double)v.lo + (double)v.hi * 18446744073709551616.0;
}
template <>
__device__ __forceinline__ double to_f64<u128>(u128 v) { return (double)v.lo + (double)v.hi * 18446744073709551616.0; }

template <typename S>
__device__ __forceinline__ bool nonzero(S v) { return v != (S)0; }
template <>
__device__ __forceinline__ bool nonzero<i128>(i128 v) { return (v.lo | (uint64_t)v.hi) != 0; }
template <>
__device__ __forceinline__ bool nonzero<u128>(u128 v) { return (v.lo | v.hi) != 0; }

// ---- DECIMAL through duckdb_value_int64 / _double / _boolean (libduckdb casts by logical type).  Restated from
// DuckDB's TryCastFromDecimal: integers round half away from zero, (input + sign * 10^scale / 2) / 10^scale with
// truncating division; double is input / 10^scale when the stored integer is exact in a double (|input| <= 2^53) or
// scale == 0, else (input / 10^scale) + (input % 10^scale) / 10^scale.  UNPINNED.
__device__ const double kDoublePow10[39] = {
    1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19,
    1e20, 1e21, 1e22, 1e23, 1e24, 1e25, 1e26, 1e27, 1e28, 1e29, 1e30, 1e31, 1e32, 1e33, 1e34, 1e35, 1e36, 1e37, 1e38};
__device__ __forceinline__ int64_t pow10_i64(int scale) {
  int64_t p = 1;
  for (int k = 0; k < scale && k < 18; ++k) p *= 10;
  return p;
}
__device__ __forceinline__ __int128 pow10_i128(int scale) {
  __int128 p = 1;
  for (int k = 0; k < scale && k < 38; ++k) p *= 10;
  return p;
}
__device__ __forceinline__ __int128 as_int128(i128 v) { return ((__int128)v.hi << 64) | (__int128)(unsigned __int128)v.lo; }
__device__ __forceinline__ double int128_to_f64(__int128 x) {
  i128 v;
  v.lo = (uint64_t)x;
  v.hi = (int64_t)(x >> 64);
  return to_f64<i128>(v);
}

template <typename S>
__device__ __forceinline__ int64_t dec_to_i64(S v, int scale) {
  const int64_t power = pow10_i64(scale);
  const int64_t x = (int64_t)v;
  const int64_t rounding = (x < 0 ? -power : power) / 2;
  return (x + rounding) / power;
}
template <>
__device__ __forceinline__ int64_t dec_to_i64<i128>(i128 v, int scale) {
  const __int128 power = pow10_i128(scale);
  const __int128 x = as_int128(v);
  const __int128 rounding = (x < 0 ? -power : power) / 2;
  const __int128 q = (x + rounding) / power;
  return (q >= -(__int128)9223372036854775807ll - 1 && q <= (__int128)9223372036854775807ll) ? (int64_t)q : 0;  // out of range: the cast fails -> 0
}
template <typename S>
__device__ __forceinline__ double dec_to_f64(S v, int scale) {
  const int64_t x = (int64_t)v;
  const double dp = kDoublePow10[scale < 0 ? 0 : (scale > 38 ? 38 : scale)];
  if (scale == 0 || (x <= 9007199254740992ll && x >= -9007199254740992ll)) return (double)x / dp;
  const int64_t power = pow10_i64(scale);
  return (double)(x / power) + (double)(x % power) / dp;
}
template <>
__device__ __forceinline__ double dec_to_f64<i128>(i128 v, int scale) {
  const __int128 x = as_int128(v);
  const double dp = kDoublePow10[scale < 0 ? 0 : (scale > 38 ? 38 : scale)];
  if (scale == 0 || (x <= (__int128)9007199254740992ll && x >= -(__int128)9007199254740992ll)) return int128_to_f64(x) / dp;
  const __int128 power = pow10_i128(scale);
  return int128_to_f64(x / power) + int128_to_f64(x % power) / dp;
}

template <typename S>
__device__ __forceinline__ int32_t to_i32_sat(S v) {  // src/duckdb_parsing.mbt:203-237
  int64_t x = (int64_t)v;
  return x > 2147483647ll ? 2147483647 : (x < -2147483648ll ? (int32_t)-2147483648ll : (int32_t)x);
}
template <>
__device__ __forceinline__ int32_t to_i32_sat<uint64_t>(uint64_t v) {
  return v > 2147483647ull ? 2147483647 : (int32_t)v;
}

__device__ __forceinline__ int64_t floor_div(int64_t a, int64_t b) {
  int64_t q = a / b;
  return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}

// The reference's typed DATE goes text -> parse_date -> date_to_days
// (src/duckdb_parsing.mbt:293-338).  date_to_days only counts leap days for years in
// [1970, year), so for year < 1970 it omits every leap day in [year, 1970).  Reproduced
// bit-exactly for the 10-character dates (years 1..9999) parse_date accepts.
__device__ __forceinline__ int32_t date_ref_quirk(int32_t days) {
  // civil_from_days (proleptic Gregorian)
  int64_t z = (int64_t)days + 719468;
  int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  int64_t doe = z - era * 146097;
  int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  int64_t y = yoe + era * 400;
  int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  int64_t mp = (5 * doy + 2) / 153;
  int64_t m = mp < 10 ? mp + 3 : mp - 9;
  if (m <= 2) y += 1;
  if (y >= 1970 || y < 1 || y > 9999) return days;
  // leap years ly with y <= ly < 1970
  auto leaps_before = [](int64_t yy) { return yy / 4 - yy / 100 + yy / 400; };  // in [1, yy]
  int64_t missing = leaps_before(1969) - leaps_before(y - 1);
  return (int32_t)((int64_t)days + missing);
}

// every functor is built from dmb_fixed_job.param (only the DECIMAL casts use it: the scale)
struct CvNoParam { __device__ __forceinline__ CvNoParam(int32_t = 0) {} };
struct CvSame : CvNoParam { using CvNoParam::CvNoParam; template <typename S> __device__ __forceinline__ S operator()(S v) const { return v; } };
struct CvI64 : CvNoParam { using CvNoParam::CvNoParam; template <typename S> __device__ __forceinline__ int64_t operator()(S v) const { return to_i64<S>(v); } };
struct CvI32Trunc : CvNoParam { using CvNoParam::CvNoParam; template <typename S> __device__ __forceinline__ int32_t operator()(S v) const { return (int32_t)to_i64<S>(v); } };
struct CvF64 : CvNoParam { using CvNoParam::CvNoParam; template <typename S> __device__ __forceinline__ double operator()(S v) const { return to_f64<S>(v); } };
struct CvBoolByte : CvNoParam { using CvNoParam::CvNoParam; template <typename S> __device__ __forceinline__ uint8_t operator()(S v) const { return nonzero<S>(v) ? 1 : 0; } };
struct CvI32Sat : CvNoParam { using CvNoParam::CvNoParam; template <typename S> __device__ __forceinline__ int32_t operator()(S v) const { return to_i32_sat<S>(v); } };
struct CvDecBase { int scale; __device__ __forceinline__ CvDecBase(int32_t p = 0) : scale(p) {} };
struct CvDecI64 : CvDecBase { using CvDecBase::CvDecBase; template <typename S> __device__ __forceinline__ int64_t operator()(S v) const { return dec_to_i64<S>(v, scale); } };
struct CvDecI32Trunc : CvDecBase { using CvDecBase::CvDecBase; template <typename S> __device__ __forceinline__ int32_t operator()(S v) const { return (int32_t)dec_to_i64<S>(v, scale); } };
struct CvDecF64 : CvDecBase { using CvDecBase::CvDecBase; template <typename S> __device__ __forceinline__ double operator()(S v) const { return dec_to_f64<S>(v, scale); } };
struct CvDecBoolByte : CvDecBase { using CvDecBase::CvDecBase; template <typename S> __device__ __forceinline__ uint8_t operator()(S v) const { return dec_to_i64<S>(v, scale) != 0 ? 1 : 0; } };
struct CvI128 : CvNoParam {
  using CvNoParam::CvNoParam;
  template <typename S> __device__ __forceinline__ i128 operator()(S v) const {
    i128 r; r.lo = (uint64_t)(int64_t)v; r.hi = (int64_t)v < 0 ? -1 : 0; return r;
  }
};
struct CvTsS : CvNoParam { using CvNoParam::CvNoParam; __device__ __forceinline__ int64_t operator()(int64_t v) const { return (int64_t)((uint64_t)v * 1000000ull); } };
struct CvTsMs : CvNoParam { using CvNoParam::CvNoParam; __device__ __forceinline__ int64_t operator()(int64_t v) const { return (int64_t)((uint64_t)v * 1000ull); } };
struct CvTsNs : CvNoParam { using CvNoParam::CvNoParam; __device__ __forceinline__ int64_t operator()(int64_t v) const { return floor_div(v, 1000); } };
struct CvMdn : CvNoParam {
  using CvNoParam::CvNoParam;
  __device__ __forceinline__ month_day_nano_t operator()(interval_t v) const {
    month_day_nano_t r; r.months = v.months; r.days = v.days; r.nanos = (int64_t)((uint64_t)v.micros * 1000ull); return r;
  }
};
struct CvDateRef : CvNoParam { using CvNoParam::CvNoParam; __device__ __forceinline__ int32_t operator()(int32_t v) const { return date_ref_quirk(v); } };
// typed TIMESTAMP through the reference's parse_timestamp: quirky day number * 86400e6 + time of day
__device__ __forceinline__ int64_t ts_ref_quirk(int64_t micros) {
  const int64_t kDay = 86400000000ll;
  const int64_t days = floor_div(micros, kDay);
  if (days < -2147483648ll || days > 2147483647ll) return micros;
  const int64_t tod = micros - days * kDay;
  return (int64_t)date_ref_quirk((int32_t)days) * kDay + tod;
}
template <typename Pre>
struct CvTsRef : CvNoParam { using CvNoParam::CvNoParam; __device__ __forceinline__ int64_t operator()(int64_t v) const { return ts_ref_quirk(Pre()(v)); } };
struct CvId64 : CvNoParam { using CvNoParam::CvNoParam; __device__ __forceinline__ int64_t operator()(int64_t v) const { return v; } };

template <typename D> __device__ __forceinline__ D zero_of() { D z; memset(&z, 0, sizeof(D)); return z; }

// ------------------------------------------------------------------ phase A: one chunk's payload
// R rows move as one naturally aligned vector of max(sizeof S, sizeof D) * R = 16 bytes; four
// vectors per thread are in flight before the first is consumed.
template <typename S, typename D, typename F>
__device__ __forceinline__ void convert_chunk(const S *__restrict__ in, const uint64_t *__restrict__ mask,
                                              D *__restrict__ out, int count, F f) {
  constexpr int W = sizeof(S) > sizeof(D) ? sizeof(S) : sizeof(D);
  constexpr int R = 16 / W;
  constexpr int U = 4;
  using PS = Pack<S, R>;
  using PD = Pack<D, R>;
  const int nvec = count / R;
  const bool out_vec_ok = (reinterpret_cast<uintptr_t>(out) % sizeof(PD)) == 0;
  const PS *vin = reinterpret_cast<const PS *>(in);
  PD *vout = reinterpret_cast<PD *>(out);
  for (int base = threadIdx.x; base < nvec; base += kThreads * U) {
    PS x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      int v = base + u * kThreads;
      if (v < nvec) x[u] = ld_stream(vin + v);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      int v = base + u * kThreads;
      if (v < nvec) {
        int row = v * R;
        uint32_t bits = mask ? (uint32_t)(__ldg(mask + (row >> 6)) >> (row & 63)) : 0xffffffffu;
        PD y;
#pragma unroll
        for (int r = 0; r < R; ++r) y.v[r] = ((bits >> r) & 1u) ? (D)f(x[u].v[r]) : zero_of<D>();
        if (out_vec_ok) {
          st_stream(vout + v, y);
        } else {
#pragma unroll
          for (int r = 0; r < R; ++r) out[row + r] = y.v[r];
        }
      }
    }
  }
  for (int row = nvec * R + threadIdx.x; row < count; row += kThreads) {
    bool valid = mask ? ((__ldg(mask + (row >> 6)) >> (row & 63)) & 1ull) : true;
    out[row] = valid ? (D)f(in[row]) : zero_of<D>();
  }
}

// Narrow types (R >= 4 rows per 16-byte vector): one chunk is only 2048 / R vectors, fewer than the
// 256 * 4 the CTA keeps in flight, so G = 1024 / (2048 / R) consecutive chunks are converted as one
// index space: every thread still has four independent 16-byte loads outstanding.
template <typename S, typename D, typename F>
__device__ __forceinline__ void convert_group(const dmb_fixed_job &job, const BatchView &b, int64_t c0, int G, F f) {
  constexpr int W = sizeof(S) > sizeof(D) ? sizeof(S) : sizeof(D);
  constexpr int R = 16 / W;
  constexpr int U = kGroupU;
  constexpr int VPC = kVec / R;  // vectors per full chunk
  using PS = Pack<S, R>;
  using PD = Pack<D, R>;
  PS x[U];
  int64_t cc[U];
  int lv[U];
  bool act[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int v = threadIdx.x + u * kThreads;
    const int g = v / VPC;
    lv[u] = v - g * VPC;
    cc[u] = c0 + g;
    act[u] = g < G && cc[u] < b.nchunks && (lv[u] + 1) * R <= (int)__ldg(b.counts + cc[u]);
    if (act[u]) {
      const S *in = reinterpret_cast<const S *>(reinterpret_cast<const uint8_t *>(job.in_data) + job.vecs[cc[u]].data_off);
      x[u] = ld_stream(reinterpret_cast<const PS *>(in) + lv[u]);
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (!act[u]) continue;
    const int64_t vo = job.vecs[cc[u]].val_off;
    const int row = lv[u] * R;
    const uint32_t bits = vo >= 0 ? (uint32_t)(__ldg(job.in_validity + vo + (row >> 6)) >> (row & 63)) : 0xffffffffu;
    D *out = reinterpret_cast<D *>(job.out_values) + __ldg(b.row_off + cc[u]);
    PD y;
#pragma unroll
    for (int r = 0; r < R; ++r) y.v[r] = ((bits >> r) & 1u) ? (D)f(x[u].v[r]) : zero_of<D>();
    if ((reinterpret_cast<uintptr_t>(out) % sizeof(PD)) == 0) {
      st_stream(reinterpret_cast<PD *>(out) + lv[u], y);
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r) out[row + r] = y.v[r];
    }
  }
  // ragged ends: the < R rows after the last whole vector of each chunk
  for (int t = threadIdx.x; t < G * R; t += kThreads) {
    const int g = t / R;
    const int64_t c = c0 + g;
    if (c >= b.nchunks) break;
    const int count = (int)__ldg(b.counts + c);
    const int row = (count / R) * R + (t - g * R);
    if (row >= count) continue;
    const dmb_vec_desc vd = job.vecs[c];
    const S *in = reinterpret_cast<const S *>(reinterpret_cast<const uint8_t *>(job.in_data) + vd.data_off);
    const bool valid = vd.val_off >= 0 ? ((__ldg(job.in_validity + vd.val_off + (row >> 6)) >> (row & 63)) & 1ull) : true;
    D *out = reinterpret_cast<D *>(job.out_values) + __ldg(b.row_off + c);
    out[row] = valid ? (D)f(in[row]) : zero_of<D>();
  }
}

// BOOLEAN bytes -> Arrow bit-packed values for output tile t (tile-centric: bit offsets of short
// chunks are arbitrary).  Thread i owns output byte i of the tile = rows 8i..8i+7.
__device__ __forceinline__ void bool_bits_tile(const BatchView &b, const dmb_fixed_job &job, int64_t t) {
  const int64_t r0 = t * (int64_t)kVec + 8 * (int64_t)threadIdx.x;
  if (r0 >= b.nrows) return;
  uint8_t *out = reinterpret_cast<uint8_t *>(job.out_values) + (r0 >> 3);
  uint32_t bits;
  if (tile_is_regular(b, t)) {
    const dmb_vec_desc vd = job.vecs[t];
    const uint8_t *in = reinterpret_cast<const uint8_t *>(job.in_data) + vd.data_off;
    int local = 8 * threadIdx.x;
    uint64_t bytes = __ldcs(reinterpret_cast<const unsigned long long *>(in + local));
    bytes = (bytes | (bytes >> 1) | (bytes >> 2) | (bytes >> 3) | (bytes >> 4) | (bytes >> 5) |
             (bytes >> 6) | (bytes >> 7)) & 0x0101010101010101ull;  // any non-zero byte is true
    bits = pack8(bytes);
    if (vd.val_off >= 0) bits &= (uint32_t)reinterpret_cast<const uint8_t *>(job.in_validity + vd.val_off)[threadIdx.x];
    int64_t left = b.nrows - r0;
    if (left < 8) bits &= (1u << left) - 1u;
  } else {
    int64_t c = find_chunk(b, r0);
    bits = 0;
    for (int k = 0; k < 8 && r0 + k < b.nrows; ++k) {
      int64_t row = r0 + k;
      while (row >= __ldg(b.row_off + c + 1)) ++c;
      int local = (int)(row - __ldg(b.row_off + c));
      const uint8_t *in = reinterpret_cast<const uint8_t *>(job.in_data) + job.vecs[c].data_off;
      bool valid = chunk_valid_bits(job.in_validity, job.vecs, c, local, 1) != 0;
      if (valid && in[local] != 0) bits |= 1u << k;
    }
  }
  *out = (uint8_t)bits;
}

// ------------------------------------------------------------------ phase B: validity of tile t
// One WARP per output tile (32 bitmap words of 64 rows): a tile is a chain of dependent loads
// (geometry -> descriptor -> mask words), so a CTA runs eight tiles side by side.
__device__ __forceinline__ void validity_tile(const BatchView &b, const dmb_fixed_job &job, int64_t t,
                                              uint64_t *s_words) {
  const int64_t nwords = (b.nrows + 63) >> 6;
  const int lane = threadIdx.x & 31;
  {
    const int64_t w = t * DMB_VALIDITY_WORDS + lane;
    uint64_t word = 0;
    if (w < nwords) {
      if (tile_is_regular(b, t)) {
        int64_t vo = job.vecs[t].val_off;
        word = vo < 0 ? ~0ull : __ldcs(reinterpret_cast<const unsigned long long *>(job.in_validity + vo + lane));
        int64_t left = b.nrows - (w << 6);
        if (left < 64) word &= (1ull << left) - 1ull;
      } else {
        word = gather_valid64(b, job.in_validity, job.vecs, w << 6);
      }
      if (job.out_validity) __stcs(reinterpret_cast<unsigned long long *>(job.out_validity + w), word);
    }
    s_words[lane] = word;
    if (job.null_count) {
      int64_t left = b.nrows - (w << 6);
      int live = w < nwords ? (left < 64 ? (int)left : 64) : 0;
      int nulls = live - __popcll(word);
      nulls = __reduce_add_sync(0xffffffffu, nulls);
      if (lane == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
    }
  }
  if (job.out_valid_bytes) {  // reference form: one byte per row, 1 = valid (duckdb_native.c:2594-2606)
    __syncwarp();
#pragma unroll 2
    for (int g = lane; g < kVec / 8; g += 32) {
      const int64_t r0 = t * (int64_t)kVec + 8 * (int64_t)g;
      if (r0 < b.nrows) {
        uint32_t bits = reinterpret_cast<const uint8_t *>(s_words)[g];
        uint64_t bytes = spread8(bits);
        uint8_t *dst = job.out_valid_bytes + r0;
        if (r0 + 8 <= b.nrows) {
          __stcs(reinterpret_cast<unsigned long long *>(dst), bytes);
        } else {
          for (int k = 0; r0 + k < b.nrows; ++k) dst[k] = (uint8_t)(bytes >> (8 * k));
        }
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------ kernels
// One instantiation per conversion (own register allocation, no mega-switch); a launch covers
// every job of a run of equal ops, so a batch costs one launch per DISTINCT conversion.
enum { kKindConvert = 0, kKindBoolBits = 1, kKindValidityOnly = 2 };

// chunks per work item: enough 16-byte vectors for the 256 x 4 loads a CTA keeps in flight
template <typename S, typename D, int KIND>
struct GroupOf {
  static constexpr int W = sizeof(S) > sizeof(D) ? sizeof(S) : sizeof(D);
  static constexpr int R = 16 / W;
  // validity only: one tile per warp
  static constexpr int value = KIND == kKindValidityOnly ? kThreads / 32 : ((KIND == kKindConvert && R >= 4) ? (kThreads * kGroupU) / (kVec / R) : 1);
};

template <typename S, typename D, typename F, int KIND>
__global__ void __launch_bounds__(kThreads)
fixed_batch_kernel(const dmb_fixed_job *__restrict__ jobs, int njobs, BatchView b) {
  __shared__ uint64_t s_words[kThreads / 32][DMB_VALIDITY_WORDS];
  __shared__ dmb_fixed_job s_job;
  constexpr int G = GroupOf<S, D, KIND>::value;
  const int64_t ntiles = (b.nrows + kVec - 1) / kVec;
  const int64_t groups = (b.nchunks + G - 1) / G;
  const int64_t items = (int64_t)njobs * groups;
  int cur_job = -1;
  for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
    const int j = (int)(item / groups);
    const int64_t i0 = (item - (int64_t)j * groups) * G;
    if (j != cur_job) {  // CTA-uniform
      __syncthreads();
      if (threadIdx.x < sizeof(dmb_fixed_job) / 8)
        reinterpret_cast<uint64_t *>(&s_job)[threadIdx.x] = reinterpret_cast<const uint64_t *>(jobs + j)[threadIdx.x];
      __syncthreads();
      cur_job = j;
    }
    const dmb_fixed_job &job = s_job;
    if (KIND == kKindConvert && job.out_values) {
      if (G > 1) {
        convert_group<S, D, F>(job, b, i0, G, F(job.param));
      } else {
        const int count = (int)__ldg(b.counts + i0);
        if (count > 0) {
          const dmb_vec_desc vd = job.vecs[i0];
          const S *in = reinterpret_cast<const S *>(reinterpret_cast<const uint8_t *>(job.in_data) + vd.data_off);
          const uint64_t *mask = vd.val_off < 0 ? nullptr : job.in_validity + vd.val_off;
          D *out = reinterpret_cast<D *>(job.out_values) + __ldg(b.row_off + i0);
          convert_chunk<S, D, F>(in, mask, out, count, F(job.param));
        }
      }
    }
    if (KIND == kKindBoolBits) {
      for (int64_t i = i0; i < i0 + G && i < b.nchunks; ++i)
        if (i < ntiles && job.out_values) bool_bits_tile(b, job, i);
    }
    if (job.out_validity || job.out_valid_bytes || job.null_count) {
      const int warp = threadIdx.x >> 5;
      for (int64_t i = i0 + warp; i < i0 + G && i < b.nchunks && i < ntiles; i += kThreads / 32) validity_tile(b, job, i, s_words[warp]);
    }
  }
}

typedef void (*fixed_kernel_fn)(const dmb_fixed_job *, int, BatchView);

#define DMB_FOR_NUMERIC(DST, DT, CV)                                                              \
  case DMB_OP(DMB_PHYS_BOOL, DST): return fixed_batch_kernel<uint8_t, DT, CV, kKindConvert>;      \
  case DMB_OP(DMB_PHYS_I8, DST): return fixed_batch_kernel<int8_t, DT, CV, kKindConvert>;         \
  case DMB_OP(DMB_PHYS_F32, DST): return fixed_batch_kernel<float, DT, CV, kKindConvert>;         \
  case DMB_OP(DMB_PHYS_F64, DST): return fixed_batch_kernel<double, DT, CV, kKindConvert>;        \
  DMB_FOR_INTS_NO8(DST, DT, CV)

#define DMB_FOR_INTS_NO8(DST, DT, CV)                                                             \
  case DMB_OP(DMB_PHYS_I16, DST): return fixed_batch_kernel<int16_t, DT, CV, kKindConvert>;       \
  case DMB_OP(DMB_PHYS_I32, DST): return fixed_batch_kernel<int32_t, DT, CV, kKindConvert>;       \
  case DMB_OP(DMB_PHYS_I64, DST): return fixed_batch_kernel<int64_t, DT, CV, kKindConvert>;       \
  case DMB_OP(DMB_PHYS_U8, DST): return fixed_batch_kernel<uint8_t, DT, CV, kKindConvert>;        \
  case DMB_OP(DMB_PHYS_U16, DST): return fixed_batch_kernel<uint16_t, DT, CV, kKindConvert>;      \
  case DMB_OP(DMB_PHYS_U32, DST): return fixed_batch_kernel<uint32_t, DT, CV, kKindConvert>;      \
  case DMB_OP(DMB_PHYS_U64, DST): return fixed_batch_kernel<uint64_t, DT, CV, kKindConvert>;

#define DMB_FOR_DECIMAL(DST, DT, CV)                                                              \
  case DMB_OP(DMB_PHYS_I16, DST): return fixed_batch_kernel<int16_t, DT, CV, kKindConvert>;       \
  case DMB_OP(DMB_PHYS_I32, DST): return fixed_batch_kernel<int32_t, DT, CV, kKindConvert>;       \
  case DMB_OP(DMB_PHYS_I64, DST): return fixed_batch_kernel<int64_t, DT, CV, kKindConvert>;       \
  case DMB_OP(DMB_PHYS_I128, DST): return fixed_batch_kernel<i128, DT, CV, kKindConvert>;

static fixed_kernel_fn select_kernel(int32_t op) {
  switch (op) {
    // raw copies, NULL slots zeroed
    case DMB_OP(DMB_PHYS_BOOL, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_I8, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_U8, DMB_DST_SAME): return fixed_batch_kernel<uint8_t, uint8_t, CvSame, kKindConvert>;
    case DMB_OP(DMB_PHYS_I16, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_U16, DMB_DST_SAME): return fixed_batch_kernel<uint16_t, uint16_t, CvSame, kKindConvert>;
    case DMB_OP(DMB_PHYS_I32, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_U32, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_F32, DMB_DST_SAME): return fixed_batch_kernel<uint32_t, uint32_t, CvSame, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_U64, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_F64, DMB_DST_SAME): return fixed_batch_kernel<uint64_t, uint64_t, CvSame, kKindConvert>;
    case DMB_OP(DMB_PHYS_I128, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_U128, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_INTERVAL, DMB_DST_SAME):
    case DMB_OP(DMB_PHYS_I128, DMB_DST_I128): return fixed_batch_kernel<u128, u128, CvSame, kKindConvert>;
    // reference getters (src/duckdb_native.c:2359-2546)
    DMB_FOR_NUMERIC(DMB_DST_I64, int64_t, CvI64)
    case DMB_OP(DMB_PHYS_I128, DMB_DST_I64): return fixed_batch_kernel<i128, int64_t, CvI64, kKindConvert>;
    DMB_FOR_NUMERIC(DMB_DST_I32_TRUNC, int32_t, CvI32Trunc)
    case DMB_OP(DMB_PHYS_I128, DMB_DST_I32_TRUNC): return fixed_batch_kernel<i128, int32_t, CvI32Trunc, kKindConvert>;
    case DMB_OP(DMB_PHYS_U128, DMB_DST_I64): return fixed_batch_kernel<u128, int64_t, CvI64, kKindConvert>;
    case DMB_OP(DMB_PHYS_U128, DMB_DST_I32_TRUNC): return fixed_batch_kernel<u128, int32_t, CvI32Trunc, kKindConvert>;
    DMB_FOR_NUMERIC(DMB_DST_F64, double, CvF64)
    case DMB_OP(DMB_PHYS_I128, DMB_DST_F64): return fixed_batch_kernel<i128, double, CvF64, kKindConvert>;
    case DMB_OP(DMB_PHYS_U128, DMB_DST_F64): return fixed_batch_kernel<u128, double, CvF64, kKindConvert>;
    DMB_FOR_NUMERIC(DMB_DST_BOOL_BYTE, uint8_t, CvBoolByte)
    case DMB_OP(DMB_PHYS_I128, DMB_DST_BOOL_BYTE): return fixed_batch_kernel<i128, uint8_t, CvBoolByte, kKindConvert>;
    case DMB_OP(DMB_PHYS_U128, DMB_DST_BOOL_BYTE): return fixed_batch_kernel<u128, uint8_t, CvBoolByte, kKindConvert>;
    // DECIMAL through the reference getters: cast by logical type (scale in job.param)
    DMB_FOR_DECIMAL(DMB_DST_DEC_I64, int64_t, CvDecI64)
    DMB_FOR_DECIMAL(DMB_DST_DEC_I32_TRUNC, int32_t, CvDecI32Trunc)
    DMB_FOR_DECIMAL(DMB_DST_DEC_F64, double, CvDecF64)
    DMB_FOR_DECIMAL(DMB_DST_DEC_BOOL_BYTE, uint8_t, CvDecBoolByte)
    case DMB_OP(DMB_PHYS_BOOL, DMB_DST_BOOL_BITS): return fixed_batch_kernel<uint8_t, uint8_t, CvSame, kKindBoolBits>;
    // Arrow decimal128 widen
    case DMB_OP(DMB_PHYS_I16, DMB_DST_I128): return fixed_batch_kernel<int16_t, i128, CvI128, kKindConvert>;
    case DMB_OP(DMB_PHYS_I32, DMB_DST_I128): return fixed_batch_kernel<int32_t, i128, CvI128, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_I128): return fixed_batch_kernel<int64_t, i128, CvI128, kKindConvert>;
    // typed columns
    case DMB_OP(DMB_PHYS_I8, DMB_DST_I32_SAT): return fixed_batch_kernel<int8_t, int32_t, CvI32Sat, kKindConvert>;
    DMB_FOR_INTS_NO8(DMB_DST_I32_SAT, int32_t, CvI32Sat)
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_US_FROM_S): return fixed_batch_kernel<int64_t, int64_t, CvTsS, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_US_FROM_MS): return fixed_batch_kernel<int64_t, int64_t, CvTsMs, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_US_FROM_NS): return fixed_batch_kernel<int64_t, int64_t, CvTsNs, kKindConvert>;
    case DMB_OP(DMB_PHYS_INTERVAL, DMB_DST_MONTH_DAY_NANO): return fixed_batch_kernel<interval_t, month_day_nano_t, CvMdn, kKindConvert>;
    case DMB_OP(DMB_PHYS_I32, DMB_DST_DATE_REF): return fixed_batch_kernel<int32_t, int32_t, CvDateRef, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_REF): return fixed_batch_kernel<int64_t, int64_t, CvTsRef<CvId64>, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_REF_FROM_S): return fixed_batch_kernel<int64_t, int64_t, CvTsRef<CvTsS>, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_REF_FROM_MS): return fixed_batch_kernel<int64_t, int64_t, CvTsRef<CvTsMs>, kKindConvert>;
    case DMB_OP(DMB_PHYS_I64, DMB_DST_TS_REF_FROM_NS): return fixed_batch_kernel<int64_t, int64_t, CvTsRef<CvTsNs>, kKindConvert>;
    case DMB_OP_VALIDITY_ONLY: return fixed_batch_kernel<uint8_t, uint8_t, CvSame, kKindValidityOnly>;
    default: return nullptr;
  }
}

// byte-per-row validity (MoonBit Array[Bool]) -> per-chunk uint64 masks, one ballot per 32 rows.
// Chunk k of the reverse path is rows [2048k, 2048k+2048), so mask words are simply word w of
// the whole bitmap; each warp produces 32-bit halves with __ballot_sync.
__global__ void __launch_bounds__(kThreads)
valid_bytes_to_masks_kernel(const uint8_t *__restrict__ valid, uint32_t *__restrict__ out32,
                            unsigned long long *null_count, int64_t nrows) {
  const int64_t nhalf = (nrows + 31) >> 5;  // 32-bit halves that contain live rows
  const int64_t nhalf_total = ((nrows + 63) >> 6) << 1;
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kThreads) >> 5;
  int nulls = 0;
  for (int64_t h = warp; h < nhalf_total; h += nwarps) {
    int64_t row = (h << 5) + lane;
    bool live = h < nhalf && row < nrows;
    bool v = live ? (__ldcs(valid + row) != 0) : false;
    uint32_t word = __ballot_sync(0xffffffffu, v);
    if (lane == 0) out32[h] = word;
    nulls += (live && !v) ? 1 : 0;
  }
  if (null_count) {
    nulls = __reduce_add_sync(0xffffffffu, nulls);
    if (lane == 0 && nulls) atomicAdd(null_count, (unsigned long long)nulls);
  }
}

}  // namespace dmb

using namespace dmb;

extern "C" int32_t dmb_dev_fixed_batch(const dmb_fixed_job *jobs_dev, const dmb_fixed_job *jobs_host,
                                       int32_t njobs, const uint32_t *counts, const int64_t *row_off,
                                       int64_t nchunks, int64_t nrows, void *stream) {
  if (njobs <= 0 || nchunks <= 0 || nrows <= 0) return 0;
  if (!jobs_dev || !jobs_host) { set_error("dmb_dev_fixed_batch: jobs is null"); return -1; }
  BatchView b{counts, row_off, nchunks, nrows};
  const int64_t max_grid = (int64_t)kNumSMs * 8;  // 8 resident CTAs of 256 threads per SM
  for (int32_t j0 = 0; j0 < njobs;) {
    int32_t j1 = j0 + 1;
    while (j1 < njobs && jobs_host[j1].op == jobs_host[j0].op) ++j1;
    fixed_kernel_fn fn = select_kernel(jobs_host[j0].op);
    if (!fn) { set_error("dmb_dev_fixed_batch: unsupported conversion op 0x%x (job %d)", jobs_host[j0].op, j0); return -1; }
    int group = 1;  // must match GroupOf<>: narrow conversions take several chunks per item
    if (jobs_host[j0].op == DMB_OP_VALIDITY_ONLY) group = kThreads / 32;  // one tile per warp
    else if ((jobs_host[j0].op & 0xff) != DMB_DST_BOOL_BITS) {
      const int wi = dmb_phys_width(jobs_host[j0].op >> 8), wo = dmb_op_out_width(jobs_host[j0].op);
      const int w = wi > wo ? wi : wo;
      if (w > 0 && w <= 4) group = (kThreads * kGroupU) / (kVec / (16 / w));
    }
    const int64_t items = (int64_t)(j1 - j0) * ((nchunks + group - 1) / group);
    const int grid = (int)(items < max_grid ? items : max_grid);
    fn<<<grid, kThreads, 0, (cudaStream_t)stream>>>(jobs_dev + j0, j1 - j0, b);
    if (check_cuda(cudaGetLastError(), "fixed_batch_kernel launch")) return -1;
    j0 = j1;
  }
  return 0;
}

extern "C" int32_t dmb_dev_valid_bytes_to_masks(const uint8_t *valid_bytes, uint64_t *out_validity,
                                                unsigned long long *null_count, int64_t nrows,
                                                void *stream) {
  if (nrows <= 0) return 0;
  int64_t warps = (nrows + 31) / 32;
  int64_t blocks = (warps + 7) / 8;
  int64_t max_grid = (int64_t)kNumSMs * 8;
  int grid = (int)(blocks < max_grid ? blocks : max_grid);
  valid_bytes_to_masks_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(
      valid_bytes, reinterpret_cast<uint32_t *>(out_validity), null_count, nrows);
  return check_cuda(cudaGetLastError(), "valid_bytes_to_masks_kernel launch");
}

// ---- host-side op table (used by the L1 layer to validate and size outputs) ----
extern "C" int32_t dmb_op_out_width(int32_t op) {
  int phys = op >> 8, dst = op & 0xff;
  static const int phys_w[DMB_PHYS_COUNT] = {1, 1, 2, 4, 8, 1, 2, 4, 8, 4, 8, 16, 16, 16, 16};
  if (phys < 0 || phys >= DMB_PHYS_STRING) return -1;
  bool numeric = phys <= DMB_PHYS_F64;
  bool integer = phys >= DMB_PHYS_I8 && phys <= DMB_PHYS_U64;
  bool huge = phys == DMB_PHYS_I128 || phys == DMB_PHYS_U128;  // HUGEINT / UHUGEINT
  bool decimal = phys == DMB_PHYS_I16 || phys == DMB_PHYS_I32 || phys == DMB_PHYS_I64 || phys == DMB_PHYS_I128;
  switch (dst) {
    case DMB_DST_SAME: return phys_w[phys];
    case DMB_DST_I32_TRUNC: return (numeric || huge) ? 4 : -1;
    case DMB_DST_I64: return (numeric || huge) ? 8 : -1;
    case DMB_DST_F64: return (numeric || huge) ? 8 : -1;
    case DMB_DST_BOOL_BYTE: return (numeric || huge) ? 1 : -1;
    case DMB_DST_DEC_I32_TRUNC: return decimal ? 4 : -1;
    case DMB_DST_DEC_I64: return decimal ? 8 : -1;
    case DMB_DST_DEC_F64: return decimal ? 8 : -1;
    case DMB_DST_DEC_BOOL_BYTE: return decimal ? 1 : -1;
    case DMB_DST_BOOL_BITS: return phys == DMB_PHYS_BOOL ? 0 : -1;
    case DMB_DST_I128:
      return (phys == DMB_PHYS_I16 || phys == DMB_PHYS_I32 || phys == DMB_PHYS_I64 || phys == DMB_PHYS_I128) ? 16 : -1;
    case DMB_DST_I32_SAT: return integer ? 4 : -1;
    case DMB_DST_TS_US_FROM_S:
    case DMB_DST_TS_US_FROM_MS:
    case DMB_DST_TS_US_FROM_NS:
    case DMB_DST_TS_REF:
    case DMB_DST_TS_REF_FROM_S:
    case DMB_DST_TS_REF_FROM_MS:
    case DMB_DST_TS_REF_FROM_NS: return phys == DMB_PHYS_I64 ? 8 : -1;
    case DMB_DST_MONTH_DAY_NANO: return phys == DMB_PHYS_INTERVAL ? 16 : -1;
    case DMB_DST_DATE_REF: return phys == DMB_PHYS_I32 ? 4 : -1;
    default: return -1;
  }
}

extern "C" int32_t dmb_phys_width(int32_t phys) {
  static const int phys_w[DMB_PHYS_COUNT] = {1, 1, 2, 4, 8, 1, 2, 4, 8, 4, 8, 16, 16, 16, 16};
  return (phys < 0 || phys >= DMB_PHYS_COUNT) ? -1 : phys_w[phys];
}
